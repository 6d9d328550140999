// group_norm.cu -- GroupNorm on NCHW fp32 maps with the pixel decoder's epilogues fused in.
//
// SURVEY.md 8f.4: around the encoder, MSDeformAttnPixelDecoder.forward_features normalises five
// feature maps with GroupNorm(32, conv_dim): the three input projections (msdeformattn.py:233-248,
// :341-345) and, at stride 4, the lateral and the output convolution of the FPN level
// (msdeformattn.py:286-300, :369-379), where it also adds the bilinearly up-sampled coarser map to
// the lateral (`y = cur + F.interpolate(out[-1], size=cur.shape[-2:], mode="bilinear",
// align_corners=False)`) and applies ReLU after the output convolution.  In torch eager that is a
// moments kernel + an elementwise kernel per GroupNorm, an up-sampling kernel and an add: at
// BASELINE configs[2] (two 1 GB maps at stride 4) 4.0 + 2.1 + 0.4 ms of a 36 ms decoder forward,
// all of it HBM-bound work running at a fraction of the roofline.
//
// Here: two launches per map.
//   1. group_stats_kernel   per (image, group) chunk -- contiguous in NCHW -- kSplit CTAs each sum
//                           (x - K) and (x - K)^2 over their part (K = the chunk's first element:
//                           the shifted sums keep E[x^2] - E[x]^2 from cancelling), in fp32 per
//                           thread over a few thousand elements, combined in fp64;
//   2. group_apply_kernel   y = (x - mean) * rstd * gamma[c] + beta[c]  [ReLU]  [+ up-sampled src],
//                           one pass, 128-bit accesses; the kSplit partials of the group are
//                           combined by every CTA itself (no atomics: deterministic).
// Algorithmic bytes: read x twice + write y once = 12 B per element (+ 1/4 of a read for the
// up-sampled map); torch's sequence moves 12 (GroupNorm) + 4 + 12 (up-sample, add) = 28.
//
// Training: the same two launches also write (mean, rstd) per (image, group) when asked (y unchanged), and the
// backward below takes three launches (reduce, per-group finalize, apply; a fourth for the gradient of the
// up-sampled map): 20 B per element (+ 5 B for that gradient) against torch's ~40.  The reference semantics are
// torch.nn.functional.group_norm and F.interpolate(mode="bilinear", align_corners=False), with torch autograd's
// gradients.
//
// Mixed precision (torch.autocast, DESIGN.md 11.3): the same kernels on a bf16 / fp16 map, widened on load, with the
// fp32 kernels' element grouping, so every fp32 result is theirs on the widened map; the 16-bit outputs (y16, grad_x)
// are those results rounded once.
#include <cuda_runtime.h>
#include <cstdint>

#include "msda_common.cuh"

namespace msda {

namespace {

constexpr int kGnSplit = 16;       // CTAs per (image, group) chunk in the statistics pass
constexpr int kGnThreads = 512;

// Element type V of the map x and of the 16-bit outputs: float, or bf16 / fp16 under torch.autocast (DESIGN.md 11.3).
// Every kernel body below is a template over it (the fp32 kernels instantiate V = float).  A thread keeps the fp32
// kernels' grouping of 4 consecutive elements -- one chunk, 16 bytes in fp32 and 8 in 16-bit -- widens on load and
// rounds once at a 16-bit store, so every fp32 sum and result is the fp32 kernel's on the widened map.
template <typename V>
using Chunk = std::conditional_t<is16<V>, uint2, float4>;
template <typename V>
__device__ __forceinline__ float4 ldg_chunk(const Chunk<V> *p) {
    if constexpr (!is16<V>) return ldg_stream_f4(p);
    else return ldg_stream_v4<V>(reinterpret_cast<const V *>(p));
}
template <typename V>
__device__ __forceinline__ void st_chunk(Chunk<V> *p, float4 o) {
    if constexpr (!is16<V>) *p = o;
    else st_round4(reinterpret_cast<V *>(p), o);
}
// one element through the read-only path, widened
template <typename V>
__device__ __forceinline__ float ldg_widen(const V *p) { return widen<float>(__ldg(p)); }

// CBIAS: a per-channel constant (the bias of the convolution that produced x, left out of that
// convolution's epilogue) is added to x on the fly: group_norm(x + cbias[c])
template <typename V, bool CBIAS>
__device__ __forceinline__ void group_stats_body(const V *__restrict__ x, double *__restrict__ partial,
                                                 long long chunk /* elements */, const float *__restrict__ cbias,
                                                 int groups, int cpg, unsigned hw4 /* chunks per channel plane */) {
    // blockIdx.x = (image * groups + group), blockIdx.y = part
    const V *base = x + (long long)blockIdx.x * chunk;
    const long long chunk4 = chunk >> 2;
    const long long per = (chunk4 + gridDim.y - 1) / gridDim.y;
    const long long beg = (long long)blockIdx.y * per, end = min(beg + per, chunk4);
    const float *cb = CBIAS ? cbias + (blockIdx.x % (unsigned)groups) * cpg : nullptr;   // the group's first channel
    const float K = ldg_widen(base) + (CBIAS ? __ldg(cb) : 0.f);
    float s = 0.f, q = 0.f;
    const Chunk<V> *b4 = reinterpret_cast<const Chunk<V> *>(base);
    for (long long i = beg + threadIdx.x; i < end; i += kGnThreads) {
        const float4 v = ldg_chunk<V>(b4 + i);
        const float Kc = CBIAS ? K - __ldg(cb + (unsigned)i / hw4) : K;      // (x + b_c) - K
        const float a = v.x - Kc, b = v.y - Kc, c = v.z - Kc, d = v.w - Kc;
        s += (a + b) + (c + d);
        q = fmaf(a, a, fmaf(b, b, fmaf(c, c, fmaf(d, d, q))));
    }
    double ds = (double)s, dq = (double)q;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        ds += __shfl_xor_sync(kFullMask, ds, o);
        dq += __shfl_xor_sync(kFullMask, dq, o);
    }
    __shared__ double ws[kGnThreads / 32], wq[kGnThreads / 32];
    if ((threadIdx.x & 31) == 0) { ws[threadIdx.x >> 5] = ds; wq[threadIdx.x >> 5] = dq; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0.0, b = 0.0;
        for (int w = 0; w < kGnThreads / 32; ++w) { a += ws[w]; b += wq[w]; }
        double *out = partial + ((long long)blockIdx.x * gridDim.y + blockIdx.y) * 2;
        out[0] = a;
        out[1] = b;
    }
}

template <bool CBIAS>
__global__ void __launch_bounds__(kGnThreads)
group_stats_kernel(const float *__restrict__ x, double *__restrict__ partial, long long chunk /* elements */,
                   const float *__restrict__ cbias, int groups, int cpg, unsigned hw4 /* float4 per channel plane */) {
    group_stats_body<float, CBIAS>(x, partial, chunk, cbias, groups, cpg, hw4);
}

template <typename V, bool CBIAS>
__global__ void __launch_bounds__(kGnThreads)
group_stats_mixed_kernel(const V *__restrict__ x, double *__restrict__ partial, long long chunk,
                         const float *__restrict__ cbias, int groups, int cpg, unsigned hw4) {
    group_stats_body<V, CBIAS>(x, partial, chunk, cbias, groups, cpg, hw4);
}

// the apply kernels' per-channel affine y = x * sc + sf (before the ReLU).  The backward rebuilds the ReLU mask
// from this very expression on the (mean, rstd) the forward wrote, so that it matches the forward bit for bit.
__device__ __forceinline__ void gn_affine(float rstd, float gamma, float beta, float cbias, float mean, float &sc,
                                          float &sf) {
    sc = rstd * gamma;
    sf = beta + (cbias - mean) * sc;
}

// Both apply kernels' first step: (mean, rstd) of group ng (= image * groups + group; N * groups fits 32 bits) from
// the kGnSplit partials of the statistics pass, and channel c's affine (sc, sf).  With mean_rstd, the CTA of the
// group's first channel and first part (blockIdx.y == 0 in both kernels) also stores (mean, rstd): one writer per group.
template <typename V>
__device__ __forceinline__ void gn_finalize(const double *__restrict__ partial, const V *__restrict__ x,
                                            const float *__restrict__ cbias, const float *__restrict__ gamma,
                                            const float *__restrict__ beta, int ng, int groups, int cpg, long long hw,
                                            float eps, int c, float *__restrict__ mean_rstd, float &sc, float &sf) {
    double a = 0.0, b = 0.0;
    const double *p = partial + (long long)ng * kGnSplit * 2;
    for (int k = 0; k < kGnSplit; ++k) { a += p[2 * k]; b += p[2 * k + 1]; }
    const double n = (double)cpg * (double)hw;
    const int g0 = (ng % groups) * cpg;                                  // the group's first channel
    const double K = (double)(ldg_widen(x + (long long)ng * cpg * hw) + (cbias ? __ldg(cbias + g0) : 0.f));
    const double mean_k = a / n;                                         // mean of (x + cbias - K)
    double var = b / n - mean_k * mean_k;
    var = var < 0.0 ? 0.0 : var;
    const float mean = (float)(mean_k + K);
    const float rstd = (float)(1.0 / sqrt(var + (double)eps));
    gn_affine(rstd, gamma[c], beta[c], cbias ? __ldg(cbias + c) : 0.f, mean, sc, sf);
    if (mean_rstd != nullptr && blockIdx.y == 0 && c == g0) {
        mean_rstd[2 * ng] = mean;
        mean_rstd[2 * ng + 1] = rstd;
    }
}

// source index of torch's bilinear up-sampling with align_corners=False
// (area_pixel_compute_source_index: scale * (dst + 0.5) - 0.5, clamped at 0)
__device__ __forceinline__ void up_index(int dst, float scale, int in_size, int &i0, int &i1, float &l1) {
    float src = scale * ((float)dst + 0.5f) - 0.5f;
    src = src < 0.f ? 0.f : src;
    i0 = min((int)src, in_size - 1);
    i1 = min(i0 + 1, in_size - 1);
    l1 = src - (float)i0;
}

// y (fp32) and, for 16-bit V, y16 (its copy rounded to V); the mixed kernels take either or both, the fp32 ones y
template <typename V, bool RELU, bool UP>
__device__ __forceinline__ void group_apply_body(const V *__restrict__ x, const double *__restrict__ partial,
                                                 const float *__restrict__ gamma, const float *__restrict__ beta,
                                                 float *__restrict__ y, V *__restrict__ y16, int C, int H, int W,
                                                 int cpg, float eps, const float *__restrict__ up, int uh, int uw,
                                                 float sh, float sw, const float *__restrict__ cbias,
                                                 float *__restrict__ mean_rstd) {
    // blockIdx.x = image * C + channel (one plane), blockIdx.y = part of the plane
    const int plane = blockIdx.x, c = plane % C;
    __shared__ float s_scale, s_shift;
    if (threadIdx.x == 0)
        gn_finalize(partial, x, cbias, gamma, beta, plane / cpg, C / cpg, cpg, (long long)H * W, eps, c, mean_rstd,
                    s_scale, s_shift);
    __syncthreads();
    const float sc = s_scale, sf = s_shift;
    const long long hw4 = ((long long)H * W) >> 2;
    const long long per = (hw4 + gridDim.y - 1) / gridDim.y;
    const long long beg = (long long)blockIdx.y * per, end = min(beg + per, hw4);
    const Chunk<V> *x4 = reinterpret_cast<const Chunk<V> *>(x) + (long long)plane * hw4;
    float4 *y4 = reinterpret_cast<float4 *>(y) + (long long)plane * hw4;
    Chunk<V> *o16 = reinterpret_cast<Chunk<V> *>(y16) + (long long)plane * hw4;
    const float *uplane = UP ? up + (long long)plane * uh * uw : nullptr;
    const int w4 = W >> 2;
    for (long long i = beg + threadIdx.x; i < end; i += 256) {
        const float4 v = ldg_chunk<V>(x4 + i);
        float4 o = make_float4(fmaf(v.x, sc, sf), fmaf(v.y, sc, sf), fmaf(v.z, sc, sf), fmaf(v.w, sc, sf));
        if (RELU) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
        if (UP) {
            const int row = (int)(i / w4), col = (int)(i - (long long)row * w4) * 4;
            int y0, y1;
            float ly;
            up_index(row, sh, uh, y0, y1, ly);
            const float *r0 = uplane + (long long)y0 * uw, *r1 = uplane + (long long)y1 * uw;
            float add[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                int x0, x1;
                float lx;
                up_index(col + k, sw, uw, x0, x1, lx);
                const float top = fmaf(lx, __ldg(r0 + x1), (1.f - lx) * __ldg(r0 + x0));
                const float bot = fmaf(lx, __ldg(r1 + x1), (1.f - lx) * __ldg(r1 + x0));
                add[k] = fmaf(ly, bot, (1.f - ly) * top);
            }
            o.x += add[0]; o.y += add[1]; o.z += add[2]; o.w += add[3];
        }
        if constexpr (!is16<V>) {
            y4[i] = o;
        } else {
            if (y != nullptr) y4[i] = o;
            if (y16 != nullptr) st_chunk<V>(o16 + i, o);
        }
    }
}

template <bool RELU, bool UP>
__global__ void __launch_bounds__(256)
group_apply_kernel(const float *__restrict__ x, const double *__restrict__ partial, const float *__restrict__ gamma,
                   const float *__restrict__ beta, float *__restrict__ y, int C, int H, int W, int cpg, float eps,
                   const float *__restrict__ up, int uh, int uw, float sh, float sw,
                   const float *__restrict__ cbias, float *__restrict__ mean_rstd) {
    group_apply_body<float, RELU, UP>(x, partial, gamma, beta, y, nullptr, C, H, W, cpg, eps, up, uh, uw, sh, sw, cbias,
                                      mean_rstd);
}

template <typename V, bool RELU, bool UP>
__global__ void __launch_bounds__(256)
group_apply_mixed_kernel(const V *__restrict__ x, const double *__restrict__ partial, const float *__restrict__ gamma,
                         const float *__restrict__ beta, float *__restrict__ y, V *__restrict__ y16, int C, int H,
                         int W, int cpg, float eps, const float *__restrict__ up, int uh, int uw, float sh, float sw,
                         const float *__restrict__ cbias, float *__restrict__ mean_rstd) {
    group_apply_body<V, RELU, UP>(x, partial, gamma, beta, y, y16, C, H, W, cpg, eps, up, uh, uw, sh, sw, cbias,
                                  mean_rstd);
}

// The same normalisation written as ROWS: y_rows[n][pixel][c] (row = the C channels of one pixel, `row_stride`
// floats apart, images `image_stride` floats apart) -- the layout the deformable encoder consumes
// (`src.flatten(2).transpose(1, 2)`, msdeformattn.py:72-79), so that the per-level maps land directly in
// their slice of the concatenated [N, S, C] tensor and torch's transposing `cat` (one more read and write of
// every map) disappears.  One CTA = 32 channels x a range of pixels; a warp turns 32 x 32 tiles through shared
// memory: 128-byte reads along the pixels of one channel, 128-bit stores along the channels of one pixel.
constexpr int kRowsWarps = 8;
constexpr int kRowsTilesPerWarp = 4;      // 32-pixel tiles per warp and CTA

__global__ void __launch_bounds__(kRowsWarps * 32)
group_apply_rows_kernel(const float *__restrict__ x, const double *__restrict__ partial, const float *__restrict__ gamma,
                        const float *__restrict__ beta, float *__restrict__ y, int C, long long hw, int cpg, float eps,
                        const float *__restrict__ cbias, long long row_stride, long long image_stride, int relu,
                        float *__restrict__ mean_rstd) {
    // blockIdx.x = image * (C / 32) + channel block, blockIdx.y = pixel range
    __shared__ float s_scale[32], s_shift[32];
    __shared__ float s_tile[kRowsWarps][32 * 33];
    const int cblocks = C / 32, n = blockIdx.x / cblocks, c0 = (blockIdx.x % cblocks) * 32;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x < 32) {
        const int c = c0 + threadIdx.x;
        gn_finalize(partial, x, cbias, gamma, beta, n * (C / cpg) + c / cpg, C / cpg, cpg, hw, eps, c, mean_rstd,
                    s_scale[threadIdx.x], s_shift[threadIdx.x]);
    }
    __syncthreads();
    float *tile = s_tile[warp];
    const float *xin = x + ((long long)n * C + c0) * hw;               // channel c0 of image n
    float *yout = y + (long long)n * image_stride + c0;
    const int sub = lane >> 3, ch4 = (lane & 7) * 4;
    const long long first = ((long long)blockIdx.y * kRowsWarps + warp) * kRowsTilesPerWarp;
    for (int t = 0; t < kRowsTilesPerWarp; ++t) {
        const long long p0 = (first + t) * 32;
        if (p0 >= hw) break;
        const long long p = p0 + lane;
#pragma unroll 8
        for (int j = 0; j < 32; ++j) {
            const float v = p < hw ? ldg_stream_f1(xin + (long long)j * hw + p) : 0.f;
            float o = fmaf(v, s_scale[j], s_shift[j]);
            if (relu) o = fmaxf(o, 0.f);
            tile[j * 33 + lane] = o;
        }
        __syncwarp();
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int pix = i * 4 + sub;
            const float4 o = make_float4(tile[(ch4 + 0) * 33 + pix], tile[(ch4 + 1) * 33 + pix],
                                         tile[(ch4 + 2) * 33 + pix], tile[(ch4 + 3) * 33 + pix]);
            if (p0 + pix < hw) *reinterpret_cast<float4 *>(yout + (p0 + pix) * row_stride + ch4) = o;
        }
        __syncwarp();
    }
}

// The same for a 16-bit x.  Sharing one body with the fp32 kernel changed that kernel's instruction schedule, so the
// fp32 source above stays as it was and this repeats it (DESIGN.md 11.3); so do the up-sampling and rows backwards.
template <typename V>
__global__ void __launch_bounds__(kRowsWarps * 32)
group_apply_rows_mixed_kernel(const V *__restrict__ x, const double *__restrict__ partial,
                              const float *__restrict__ gamma, const float *__restrict__ beta, float *__restrict__ y,
                              int C, long long hw, int cpg, float eps, const float *__restrict__ cbias,
                              long long row_stride, long long image_stride, int relu, float *__restrict__ mean_rstd) {
    // blockIdx.x = image * (C / 32) + channel block, blockIdx.y = pixel range
    __shared__ float s_scale[32], s_shift[32];
    __shared__ float s_tile[kRowsWarps][32 * 33];
    const int cblocks = C / 32, n = blockIdx.x / cblocks, c0 = (blockIdx.x % cblocks) * 32;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x < 32) {
        const int c = c0 + threadIdx.x;
        gn_finalize(partial, x, cbias, gamma, beta, n * (C / cpg) + c / cpg, C / cpg, cpg, hw, eps, c, mean_rstd,
                    s_scale[threadIdx.x], s_shift[threadIdx.x]);
    }
    __syncthreads();
    float *tile = s_tile[warp];
    const V *xin = x + ((long long)n * C + c0) * hw;                   // channel c0 of image n
    float *yout = y + (long long)n * image_stride + c0;
    const int sub = lane >> 3, ch4 = (lane & 7) * 4;
    const long long first = ((long long)blockIdx.y * kRowsWarps + warp) * kRowsTilesPerWarp;
    for (int t = 0; t < kRowsTilesPerWarp; ++t) {
        const long long p0 = (first + t) * 32;
        if (p0 >= hw) break;
        const long long p = p0 + lane;
#pragma unroll 8
        for (int j = 0; j < 32; ++j) {
            const float v = p < hw ? ldg_stream_one<V>(xin + (long long)j * hw + p) : 0.f;
            float o = fmaf(v, s_scale[j], s_shift[j]);
            if (relu) o = fmaxf(o, 0.f);
            tile[j * 33 + lane] = o;
        }
        __syncwarp();
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int pix = i * 4 + sub;
            const float4 o = make_float4(tile[(ch4 + 0) * 33 + pix], tile[(ch4 + 1) * 33 + pix],
                                         tile[(ch4 + 2) * 33 + pix], tile[(ch4 + 3) * 33 + pix]);
            if (p0 + pix < hw) *reinterpret_cast<float4 *>(yout + (p0 + pix) * row_stride + ch4) = o;
        }
        __syncwarp();
    }
}



// What the NCHW kernels need, forward and backward: planes walked as float4 (H*W % 4 == 0; W % 4 == 0 as well with
// the up-sampled map, whose add takes 4 outputs of one row), 32-bit plane and chunk counts, and 16-byte aligned maps
// (`maps`: their addresses or-ed together)
bool gn_nchw_ok(int N, int C, int H, int W, int groups, bool up, uintptr_t maps) {
    const long long hw = (long long)H * W;
    return groups > 0 && C % groups == 0 && !(hw & 3) && !(up && (W & 3)) && hw <= 0x7fffffffLL &&
           (long long)N * C <= 0x7fffffffLL && (long long)N * groups <= 0x7fffffffLL && !(maps & 15u);
}

// pixel ranges of the rows kernels' apply grid (blockIdx.y)
long long gn_rows_parts(long long hw) {
    const long long per_cta = 32LL * kRowsWarps * kRowsTilesPerWarp;
    return (hw + per_cta - 1) / per_cta;
}

// What the rows kernels need, forward and backward: 32-channel blocks, planes of whole float4, rows of whole float4
// (row and image strides), 16-byte aligned maps and rows (`maps`), and at most 65535 pixel ranges
bool gn_rows_ok(int N, int C, long long hw, int groups, long long row_stride, long long image_stride, uintptr_t maps) {
    return groups > 0 && C % groups == 0 && C % 32 == 0 && !(hw & 3) && hw <= 0x7fffffffLL && row_stride >= C &&
           !(row_stride & 3) && !(image_stride & 3) && (long long)N * (C / 32) <= 0x7fffffffLL &&
           (long long)N * groups <= 0x7fffffffLL && !(maps & 15u) && gn_rows_parts(hw) <= 65535;
}

uintptr_t addr(const void *p) { return reinterpret_cast<uintptr_t>(p); }
// the address bits of a map that must be zero, or-ed into the `maps` of gn_nchw_ok / gn_rows_ok: 16-byte alignment
// for an fp32 map, 8-byte alignment (one chunk) for a 16-bit one; NULL passes
template <typename V>
uintptr_t amap(const V *p) { return addr(p) & (is16<V> ? 7u : 15u); }

// The first launch of both forward layouts: the kGnSplit partial sums of every (image, group) chunk of x (+ cbias).
// Sets *handled unless the chunk is too long for the CBIAS variant's 32-bit channel lookup.
template <typename V>
cudaError_t launch_group_stats(const V *x, const float *cbias, int N, int C, long long hw, int groups,
                               double *workspace, cudaStream_t stream, bool *handled) {
    const int cpg = C / groups;
    const long long chunk = (long long)cpg * hw;
    if (cbias != nullptr && chunk > 0x7fffffffLL) return cudaSuccess;
    *handled = true;
    const dim3 sgrid((unsigned)(N * groups), kGnSplit);
    if constexpr (is16<V>) {
        if (cbias != nullptr)
            group_stats_mixed_kernel<V, true><<<sgrid, kGnThreads, 0, stream>>>(x, workspace, chunk, cbias, groups, cpg, (unsigned)(hw >> 2));
        else
            group_stats_mixed_kernel<V, false><<<sgrid, kGnThreads, 0, stream>>>(x, workspace, chunk, nullptr, groups, cpg, 1u);
    } else {
        if (cbias != nullptr)
            group_stats_kernel<true><<<sgrid, kGnThreads, 0, stream>>>(x, workspace, chunk, cbias, groups, cpg, (unsigned)(hw >> 2));
        else
            group_stats_kernel<false><<<sgrid, kGnThreads, 0, stream>>>(x, workspace, chunk, nullptr, groups, cpg, 1u);
    }
    note_launch();
    return cudaGetLastError();
}

}  // namespace

// workspace: N * groups * kGnSplit * 2 doubles.  V = float: y only (y16 unused); 16-bit V: y and / or y16
template <typename V>
cudaError_t launch_group_norm(const V *x, const float *cbias, const float *gamma, const float *beta, float *y, V *y16,
                              int N, int C, int H, int W, int groups, float eps, int relu, const float *up, int uh,
                              int uw, double *workspace, float *mean_rstd, cudaStream_t stream, bool *handled) {
    *handled = false;
    if (!gn_nchw_ok(N, C, H, W, groups, up != nullptr, amap(x) | amap(y) | amap(y16)) ||
        (up != nullptr && (uh <= 0 || uw <= 0)))
        return cudaSuccess;
    const long long hw = (long long)H * W;
    cudaError_t e = launch_group_stats(x, cbias, N, C, hw, groups, workspace, stream, handled);
    if (e != cudaSuccess || !*handled) return e;
    // parts per plane: enough CTAs for the whole GPU, each with a few thousand float4
    int parts = (int)((hw / 4 + 8191) / 8192);
    if (parts < 1) parts = 1;
    if (parts > 64) parts = 64;
    const dim3 grid((unsigned)(N * C), (unsigned)parts);
    const int cpg = C / groups;
    const float sh = up ? (float)uh / (float)H : 0.f, sw = up ? (float)uw / (float)W : 0.f;
#define GN_APPLY(R, U)                                                                                                   \
    do {                                                                                                                 \
        if constexpr (is16<V>)                                                                                           \
            group_apply_mixed_kernel<V, R, U><<<grid, 256, 0, stream>>>(x, workspace, gamma, beta, y, y16, C, H, W, cpg, \
                                                                        eps, up, uh, uw, sh, sw, cbias, mean_rstd);      \
        else                                                                                                             \
            group_apply_kernel<R, U><<<grid, 256, 0, stream>>>(x, workspace, gamma, beta, y, C, H, W, cpg, eps, up, uh,  \
                                                               uw, sh, sw, cbias, mean_rstd);                            \
    } while (0)
    if (up != nullptr) { if (relu) GN_APPLY(true, true); else GN_APPLY(false, true); }
    else { if (relu) GN_APPLY(true, false); else GN_APPLY(false, false); }
#undef GN_APPLY
    note_launch();
    return cudaGetLastError();
}

// GroupNorm of x[N, C, H*W] written as fp32 rows: y[n * image_stride + pixel * row_stride + c]
template <typename V>
cudaError_t launch_group_norm_rows(const V *x, const float *cbias, const float *gamma, const float *beta, float *y,
                                   int N, int C, long long hw, int groups, float eps, int relu, long long row_stride,
                                   long long image_stride, double *workspace, float *mean_rstd, cudaStream_t stream,
                                   bool *handled) {
    *handled = false;
    if (!gn_rows_ok(N, C, hw, groups, row_stride, image_stride, amap(x) | amap(y))) return cudaSuccess;
    cudaError_t e = launch_group_stats(x, cbias, N, C, hw, groups, workspace, stream, handled);
    if (e != cudaSuccess || !*handled) return e;
    const dim3 grid((unsigned)(N * (C / 32)), (unsigned)gn_rows_parts(hw));
    if constexpr (is16<V>)
        group_apply_rows_mixed_kernel<V><<<grid, kRowsWarps * 32, 0, stream>>>(
            x, workspace, gamma, beta, y, C, hw, C / groups, eps, cbias, row_stride, image_stride, relu, mean_rstd);
    else
        group_apply_rows_kernel<<<grid, kRowsWarps * 32, 0, stream>>>(
            x, workspace, gamma, beta, y, C, hw, C / groups, eps, cbias, row_stride, image_stride, relu, mean_rstd);
    note_launch();
    return cudaGetLastError();
}

#define GN_FWD_INSTANTIATE(V)                                                                                          \
    template cudaError_t launch_group_norm<V>(const V *, const float *, const float *, const float *, float *, V *,    \
                                              int, int, int, int, int, float, int, const float *, int, int, double *,  \
                                              float *, cudaStream_t, bool *);                                          \
    template cudaError_t launch_group_norm_rows<V>(const V *, const float *, const float *, const float *, float *,     \
                                                   int, int, long long, int, float, int, long long, long long,         \
                                                   double *, float *, cudaStream_t, bool *);
GN_FWD_INSTANTIATE(float)
GN_FWD_INSTANTIATE(__nv_bfloat16)
GN_FWD_INSTANTIATE(__half)
#undef GN_FWD_INSTANTIATE

int group_norm_workspace_doubles(int N, int groups) { return N * groups * kGnSplit * 2; }

// ------------------------------------------------------------------------------------------------ backward
// With x' = x + cbias[c], xh = (x' - mean) * rstd, gy = grad_y * [ReLU mask] and m = cpg * H * W:
//   reduce:   per (n, c) plane  A = sum gy,  B = sum gy * xh,  X = sum xh                  (reads grad_y, x)
//   finalize: per (n, g)  a = sum_c gamma_c A,  b = sum_c gamma_c B;  per c  grad_beta = sum_n A,
//             grad_gamma = sum_n B,  grad_cbias = sum_n rstd * (gamma_c A - a / cpg - X b / m)  (no pass over the map)
//   apply:    grad_x = rstd * (gamma_c * gy - a / m - xh * b / m)                            (reads grad_y, x; writes grad_x)
//   up:       grad_up = the adjoint of the forward's bilinear up-sampling applied to grad_y (unmasked: the add
//             comes after the ReLU), gathered per source pixel          (reads grad_y, writes grad_up)
// Partial sums go to fixed slots and are combined in fp64 in a fixed order: no atomics, the same bits every run.
namespace {

constexpr int kBwdMaxParts = 16;          // reduce-pass CTAs per plane (NCHW) or per 32-channel block (rows)
constexpr int kBwdThreads = 256;

// per-channel constants of the backward from the forward's (mean, rstd) of group ng
struct GnChan {
    float sc, sf;                         // the forward's affine (ReLU mask)
    float mc, rstd;                       // xh = (x - mc) * rstd, mc = mean - cbias[c]
};

__device__ __forceinline__ GnChan gn_chan(const float *mean_rstd, long long ng, const float *gamma, const float *beta,
                                          const float *cbias, int c) {
    GnChan k;
    const float mean = __ldg(mean_rstd + 2 * ng), rstd = __ldg(mean_rstd + 2 * ng + 1);
    const float cb = cbias ? __ldg(cbias + c) : 0.f;
    gn_affine(rstd, __ldg(gamma + c), __ldg(beta + c), cb, mean, k.sc, k.sf);
    k.mc = mean - cb;
    k.rstd = rstd;
    return k;
}

// one element of the reduce pass
__device__ __forceinline__ void gn_bwd_acc(float v, float g, const GnChan &k, bool relu, float &sa, float &sb,
                                           float &sx) {
    const float xh = (v - k.mc) * k.rstd;
    if (relu && !(fmaf(v, k.sc, k.sf) > 0.f)) g = 0.f;
    sa += g;
    sb = fmaf(g, xh, sb);
    sx += xh;
}

// one element of the apply pass: k1 = rstd * gamma_c, ka = -rstd * a / m, kb = -rstd * b / m
__device__ __forceinline__ float gn_bwd_dx(float v, float g, const GnChan &k, bool relu, float k1, float ka, float kb) {
    const float xh = (v - k.mc) * k.rstd;
    if (relu && !(fmaf(v, k.sc, k.sf) > 0.f)) g = 0.f;
    return fmaf(k1, g, fmaf(xh, kb, ka));
}

// blockDim.x = kBwdThreads; the CTA's three sums combined in fp64 and written to slot `out`
__device__ __forceinline__ void gn_bwd_store_sums(double a, double b, double x, double *out) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(kFullMask, a, o);
        b += __shfl_xor_sync(kFullMask, b, o);
        x += __shfl_xor_sync(kFullMask, x, o);
    }
    __shared__ double red[3][kBwdThreads / 32];
    if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = a; red[1][threadIdx.x >> 5] = b; red[2][threadIdx.x >> 5] = x; }
    __syncthreads();
    if (threadIdx.x == 0) {
        a = b = x = 0.0;
        for (int w = 0; w < kBwdThreads / 32; ++w) { a += red[0][w]; b += red[1][w]; x += red[2][w]; }
        out[0] = a;
        out[1] = b;
        out[2] = x;
    }
}

// G: element type of grad_y (float, or V: the gradient of the forward's y16); V: of x (and of grad_x)
template <typename G, typename V, bool RELU>
__device__ __forceinline__ void gn_bwd_reduce_body(const G *__restrict__ gy, const V *__restrict__ x,
                                                   const float *__restrict__ mean_rstd, const float *__restrict__ gamma,
                                                   const float *__restrict__ beta, const float *__restrict__ cbias,
                                                   double *__restrict__ partial, int C, int cpg, long long hw4) {
    // blockIdx.x = image * C + channel (one plane), blockIdx.y = part of the plane
    const int plane = blockIdx.x, c = plane % C;
    const GnChan k = gn_chan(mean_rstd, plane / cpg, gamma, beta, cbias, c);
    const long long per = (hw4 + gridDim.y - 1) / gridDim.y;
    const long long beg = (long long)blockIdx.y * per, end = min(beg + per, hw4);
    const Chunk<V> *x4 = reinterpret_cast<const Chunk<V> *>(x) + (long long)plane * hw4;
    const Chunk<G> *g4 = reinterpret_cast<const Chunk<G> *>(gy) + (long long)plane * hw4;
    double da = 0.0, db = 0.0, dx = 0.0;           // fp32 within a float4, fp64 across them
    for (long long i = beg + threadIdx.x; i < end; i += kBwdThreads) {
        const float4 v = ldg_chunk<V>(x4 + i), g = ldg_chunk<G>(g4 + i);
        float sa = 0.f, sb = 0.f, sx = 0.f;
        gn_bwd_acc(v.x, g.x, k, RELU, sa, sb, sx);
        gn_bwd_acc(v.y, g.y, k, RELU, sa, sb, sx);
        gn_bwd_acc(v.z, g.z, k, RELU, sa, sb, sx);
        gn_bwd_acc(v.w, g.w, k, RELU, sa, sb, sx);
        da += (double)sa;
        db += (double)sb;
        dx += (double)sx;
    }
    gn_bwd_store_sums(da, db, dx, partial + ((long long)plane * kBwdMaxParts + blockIdx.y) * 3);
}

template <bool RELU>
__global__ void __launch_bounds__(kBwdThreads)
gn_bwd_reduce_kernel(const float *__restrict__ gy, const float *__restrict__ x, const float *__restrict__ mean_rstd,
                     const float *__restrict__ gamma, const float *__restrict__ beta, const float *__restrict__ cbias,
                     double *__restrict__ partial, int C, int cpg, long long hw4) {
    gn_bwd_reduce_body<float, float, RELU>(gy, x, mean_rstd, gamma, beta, cbias, partial, C, cpg, hw4);
}

template <typename G, typename V, bool RELU>
__global__ void __launch_bounds__(kBwdThreads)
gn_bwd_reduce_mixed_kernel(const G *__restrict__ gy, const V *__restrict__ x, const float *__restrict__ mean_rstd,
                           const float *__restrict__ gamma, const float *__restrict__ beta,
                           const float *__restrict__ cbias, double *__restrict__ partial, int C, int cpg,
                           long long hw4) {
    gn_bwd_reduce_body<G, V, RELU>(gy, x, mean_rstd, gamma, beta, cbias, partial, C, cpg, hw4);
}

// one CTA per group: the parts of every (n, c) of the group -> abx, the (n, g) sums -> ab, the parameter gradients
__global__ void __launch_bounds__(kBwdThreads)
gn_bwd_finalize_kernel(const double *__restrict__ partial, int parts, const float *__restrict__ gamma,
                       const float *__restrict__ mean_rstd, int N, int C, int cpg, long long hw,
                       double *__restrict__ abx, double *__restrict__ ab, float *__restrict__ grad_gamma,
                       float *__restrict__ grad_beta, float *__restrict__ grad_cbias) {
    const int g = blockIdx.x, groups = C / cpg;
    for (int i = threadIdx.x; i < N * cpg; i += kBwdThreads) {
        const long long plane = (long long)(i / cpg) * C + g * cpg + i % cpg;
        const double *p = partial + plane * kBwdMaxParts * 3;
        double A = 0.0, B = 0.0, X = 0.0;
        for (int k = 0; k < parts; ++k) { A += p[3 * k]; B += p[3 * k + 1]; X += p[3 * k + 2]; }
        abx[plane * 3] = A;
        abx[plane * 3 + 1] = B;
        abx[plane * 3 + 2] = X;
    }
    __syncthreads();
    for (int n = threadIdx.x; n < N; n += kBwdThreads) {
        double a = 0.0, b = 0.0;
        for (int j = 0; j < cpg; ++j) {
            const int c = g * cpg + j;
            const double *s = abx + ((long long)n * C + c) * 3;
            a += (double)gamma[c] * s[0];
            b += (double)gamma[c] * s[1];
        }
        ab[((long long)n * groups + g) * 2] = a;
        ab[((long long)n * groups + g) * 2 + 1] = b;
    }
    __syncthreads();
    const double m = (double)cpg * (double)hw;
    for (int j = threadIdx.x; j < cpg; j += kBwdThreads) {
        const int c = g * cpg + j;
        double sg = 0.0, sb = 0.0, scb = 0.0;
        for (int n = 0; n < N; ++n) {
            const double *s = abx + ((long long)n * C + c) * 3;
            const long long ng = (long long)n * groups + g;
            sb += s[0];
            sg += s[1];
            if (grad_cbias)
                scb += (double)mean_rstd[2 * ng + 1] *
                       ((double)gamma[c] * s[0] - ab[2 * ng] / cpg - s[2] * ab[2 * ng + 1] / m);
        }
        grad_gamma[c] = (float)sg;
        grad_beta[c] = (float)sb;
        if (grad_cbias) grad_cbias[c] = (float)scb;
    }
}

// the apply pass's per-channel factors from the finalized (n, g) sums
__device__ __forceinline__ void gn_bwd_factors(const GnChan &k, float gamma, const double *ab, long long ng, double m,
                                               float &k1, float &ka, float &kb) {
    k1 = k.rstd * gamma;
    ka = (float)(-(double)k.rstd * ab[2 * ng] / m);
    kb = (float)(-(double)k.rstd * ab[2 * ng + 1] / m);
}

template <typename G, typename V, bool RELU>
__device__ __forceinline__ void gn_bwd_apply_body(const G *__restrict__ gy, const V *__restrict__ x,
                                                  const float *__restrict__ mean_rstd, const float *__restrict__ gamma,
                                                  const float *__restrict__ beta, const float *__restrict__ cbias,
                                                  const double *__restrict__ ab, V *__restrict__ gx, int C, int cpg,
                                                  long long hw4) {
    // blockIdx.x = image * C + channel (one plane), blockIdx.y = part of the plane
    const int plane = blockIdx.x, c = plane % C;
    __shared__ GnChan s_k;
    __shared__ float s_f[3];
    if (threadIdx.x == 0) {
        s_k = gn_chan(mean_rstd, plane / cpg, gamma, beta, cbias, c);
        gn_bwd_factors(s_k, __ldg(gamma + c), ab, plane / cpg, (double)cpg * (double)(hw4 * 4), s_f[0], s_f[1], s_f[2]);
    }
    __syncthreads();
    const GnChan k = s_k;
    const float k1 = s_f[0], ka = s_f[1], kb = s_f[2];
    const long long per = (hw4 + gridDim.y - 1) / gridDim.y;
    const long long beg = (long long)blockIdx.y * per, end = min(beg + per, hw4);
    const Chunk<V> *x4 = reinterpret_cast<const Chunk<V> *>(x) + (long long)plane * hw4;
    const Chunk<G> *g4 = reinterpret_cast<const Chunk<G> *>(gy) + (long long)plane * hw4;
    Chunk<V> *o4 = reinterpret_cast<Chunk<V> *>(gx) + (long long)plane * hw4;
    for (long long i = beg + threadIdx.x; i < end; i += kBwdThreads) {
        const float4 v = ldg_chunk<V>(x4 + i), g = ldg_chunk<G>(g4 + i);
        st_chunk<V>(o4 + i, make_float4(gn_bwd_dx(v.x, g.x, k, RELU, k1, ka, kb), gn_bwd_dx(v.y, g.y, k, RELU, k1, ka, kb),
                                        gn_bwd_dx(v.z, g.z, k, RELU, k1, ka, kb), gn_bwd_dx(v.w, g.w, k, RELU, k1, ka, kb)));
    }
}

template <bool RELU>
__global__ void __launch_bounds__(kBwdThreads)
gn_bwd_apply_kernel(const float *__restrict__ gy, const float *__restrict__ x, const float *__restrict__ mean_rstd,
                    const float *__restrict__ gamma, const float *__restrict__ beta, const float *__restrict__ cbias,
                    const double *__restrict__ ab, float *__restrict__ gx, int C, int cpg, long long hw4) {
    gn_bwd_apply_body<float, float, RELU>(gy, x, mean_rstd, gamma, beta, cbias, ab, gx, C, cpg, hw4);
}

template <typename G, typename V, bool RELU>
__global__ void __launch_bounds__(kBwdThreads)
gn_bwd_apply_mixed_kernel(const G *__restrict__ gy, const V *__restrict__ x, const float *__restrict__ mean_rstd,
                          const float *__restrict__ gamma, const float *__restrict__ beta,
                          const float *__restrict__ cbias, const double *__restrict__ ab, V *__restrict__ gx, int C,
                          int cpg, long long hw4) {
    gn_bwd_apply_body<G, V, RELU>(gy, x, mean_rstd, gamma, beta, cbias, ab, gx, C, cpg, hw4);
}

// destinations whose up_index names source s as i0 or i1: their source coordinate lies in [s - 1, s + 1) (for the
// last source: everything clamped onto it), i.e. dst + 0.5 in [(s - 0.5) / scale, (s + 1.5) / scale).  One index of
// slack on either side absorbs the rounding of this estimate; the exact test is up_index itself.
__device__ __forceinline__ void up_range(int s, float scale, int in_size, int out_size, int &lo, int &hi) {
    lo = max(0, (int)floorf(((float)s - 0.5f) / scale - 0.5f) - 1);
    hi = s == in_size - 1 ? out_size : min(out_size, (int)ceilf(((float)s + 1.5f) / scale - 0.5f) + 1);
}

// grad_up[plane][sy][sx] = sum over the destination pixels that read source (sy, sx), with the forward's weights
__global__ void __launch_bounds__(kBwdThreads)
gn_bwd_up_kernel(const float *__restrict__ gy, float *__restrict__ gup, int H, int W, int uh, int uw, float sh,
                 float sw) {
    // blockIdx.x = plane, blockIdx.y = range of source pixels
    const float *g = gy + (long long)blockIdx.x * H * W;
    float *o = gup + (long long)blockIdx.x * uh * uw;
    for (int s = blockIdx.y * kBwdThreads + threadIdx.x; s < uh * uw; s += gridDim.y * kBwdThreads) {
        const int sy = s / uw, sx = s - sy * uw;
        int r0, r1, q0, q1;
        up_range(sy, sh, uh, H, r0, r1);
        up_range(sx, sw, uw, W, q0, q1);
        float acc = 0.f;
        for (int dr = r0; dr < r1; ++dr) {
            int y0, y1;
            float ly;
            up_index(dr, sh, uh, y0, y1, ly);
            const float wy = (y0 == sy ? 1.f - ly : 0.f) + (y1 == sy ? ly : 0.f);
            if (y0 != sy && y1 != sy) continue;
            const float *row = g + (long long)dr * W;
            float sum = 0.f;
            for (int dc = q0; dc < q1; ++dc) {
                int x0, x1;
                float lx;
                up_index(dc, sw, uw, x0, x1, lx);
                if (x0 != sx && x1 != sx) continue;
                const float wx = (x0 == sx ? 1.f - lx : 0.f) + (x1 == sx ? lx : 0.f);
                sum = fmaf(wx, __ldg(row + dc), sum);
            }
            acc = fmaf(wy, sum, acc);
        }
        o[s] = acc;
    }
}

// the same for a 16-bit grad_y (the gradient of y16): a copy of the fp32 source (DESIGN.md 11.3)
template <typename G>
__global__ void __launch_bounds__(kBwdThreads)
gn_bwd_up_mixed_kernel(const G *__restrict__ gy, float *__restrict__ gup, int H, int W, int uh, int uw, float sh,
                       float sw) {
    // blockIdx.x = plane, blockIdx.y = range of source pixels
    const G *g = gy + (long long)blockIdx.x * H * W;
    float *o = gup + (long long)blockIdx.x * uh * uw;
    for (int s = blockIdx.y * kBwdThreads + threadIdx.x; s < uh * uw; s += gridDim.y * kBwdThreads) {
        const int sy = s / uw, sx = s - sy * uw;
        int r0, r1, q0, q1;
        up_range(sy, sh, uh, H, r0, r1);
        up_range(sx, sw, uw, W, q0, q1);
        float acc = 0.f;
        for (int dr = r0; dr < r1; ++dr) {
            int y0, y1;
            float ly;
            up_index(dr, sh, uh, y0, y1, ly);
            const float wy = (y0 == sy ? 1.f - ly : 0.f) + (y1 == sy ? ly : 0.f);
            if (y0 != sy && y1 != sy) continue;
            const G *row = g + (long long)dr * W;
            float sum = 0.f;
            for (int dc = q0; dc < q1; ++dc) {
                int x0, x1;
                float lx;
                up_index(dc, sw, uw, x0, x1, lx);
                if (x0 != sx && x1 != sx) continue;
                const float wx = (x0 == sx ? 1.f - lx : 0.f) + (x1 == sx ? lx : 0.f);
                sum = fmaf(wx, ldg_widen(row + dc), sum);
            }
            acc = fmaf(wy, sum, acc);
        }
        o[s] = acc;
    }
}



// rows layout: grad_y[n * image_stride + pixel * row_stride + c], x and grad_x NCHW.  One CTA = 32 channels x a range
// of pixels, as in the forward's rows kernel.  Reduce: a warp stages a 32-channel x 32-pixel tile of x in shared
// memory and each lane (= one channel) walks the pixels, reading grad_y along the channels of one pixel (128 bytes
// per warp load).
__global__ void __launch_bounds__(kRowsWarps * 32)
gn_bwd_rows_reduce_kernel(const float *__restrict__ gy, long long row_stride, long long image_stride,
                          const float *__restrict__ x, const float *__restrict__ mean_rstd,
                          const float *__restrict__ gamma, const float *__restrict__ beta,
                          const float *__restrict__ cbias, double *__restrict__ partial, int C, long long hw, int cpg,
                          int relu) {
    // blockIdx.x = image * (C / 32) + channel block, blockIdx.y = part
    __shared__ float s_tile[kRowsWarps][32 * 33];
    __shared__ double s_red[3][kRowsWarps][32];
    const int cblocks = C / 32, n = blockIdx.x / cblocks, c0 = (blockIdx.x % cblocks) * 32;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, c = c0 + lane;
    const GnChan k = gn_chan(mean_rstd, (long long)n * (C / cpg) + c / cpg, gamma, beta, cbias, c);
    float *tile = s_tile[warp];
    const float *xin = x + ((long long)n * C + c0) * hw;
    const float *gin = gy + (long long)n * image_stride + c;
    double da = 0.0, db = 0.0, dx = 0.0;           // fp32 within a tile, fp64 across tiles
    for (long long t = (long long)blockIdx.y * kRowsWarps + warp; t * 32 < hw; t += (long long)gridDim.y * kRowsWarps) {
        const long long p0 = t * 32, p = p0 + lane;
#pragma unroll 8
        for (int j = 0; j < 32; ++j) tile[j * 33 + lane] = p < hw ? ldg_stream_f1(xin + (long long)j * hw + p) : 0.f;
        __syncwarp();
        const int np = (int)min(32LL, hw - p0);
        float sa = 0.f, sb = 0.f, sx = 0.f;
        for (int q = 0; q < np; ++q)
            gn_bwd_acc(tile[lane * 33 + q], ldg_stream_f1(gin + (p0 + q) * row_stride), k, relu != 0, sa, sb, sx);
        da += (double)sa;
        db += (double)sb;
        dx += (double)sx;
        __syncwarp();
    }
    s_red[0][warp][lane] = da;
    s_red[1][warp][lane] = db;
    s_red[2][warp][lane] = dx;
    __syncthreads();
    if (warp == 0) {
        double a = 0.0, b = 0.0, xs = 0.0;
        for (int w = 0; w < kRowsWarps; ++w) { a += s_red[0][w][lane]; b += s_red[1][w][lane]; xs += s_red[2][w][lane]; }
        double *out = partial + (((long long)n * C + c) * kBwdMaxParts + blockIdx.y) * 3;
        out[0] = a;
        out[1] = b;
        out[2] = xs;
    }
}

// the same for a 16-bit x: a copy of the fp32 source (DESIGN.md 11.3)
template <typename V>
__global__ void __launch_bounds__(kRowsWarps * 32)
gn_bwd_rows_reduce_mixed_kernel(const float *__restrict__ gy, long long row_stride, long long image_stride,
                                const V *__restrict__ x, const float *__restrict__ mean_rstd,
                                const float *__restrict__ gamma, const float *__restrict__ beta,
                                const float *__restrict__ cbias, double *__restrict__ partial, int C, long long hw,
                                int cpg, int relu) {
    // blockIdx.x = image * (C / 32) + channel block, blockIdx.y = part
    __shared__ float s_tile[kRowsWarps][32 * 33];
    __shared__ double s_red[3][kRowsWarps][32];
    const int cblocks = C / 32, n = blockIdx.x / cblocks, c0 = (blockIdx.x % cblocks) * 32;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, c = c0 + lane;
    const GnChan k = gn_chan(mean_rstd, (long long)n * (C / cpg) + c / cpg, gamma, beta, cbias, c);
    float *tile = s_tile[warp];
    const V *xin = x + ((long long)n * C + c0) * hw;
    const float *gin = gy + (long long)n * image_stride + c;
    double da = 0.0, db = 0.0, dx = 0.0;           // fp32 within a tile, fp64 across tiles
    for (long long t = (long long)blockIdx.y * kRowsWarps + warp; t * 32 < hw; t += (long long)gridDim.y * kRowsWarps) {
        const long long p0 = t * 32, p = p0 + lane;
#pragma unroll 8
        for (int j = 0; j < 32; ++j) tile[j * 33 + lane] = p < hw ? ldg_stream_one<V>(xin + (long long)j * hw + p) : 0.f;
        __syncwarp();
        const int np = (int)min(32LL, hw - p0);
        float sa = 0.f, sb = 0.f, sx = 0.f;
        for (int q = 0; q < np; ++q)
            gn_bwd_acc(tile[lane * 33 + q], ldg_stream_f1(gin + (p0 + q) * row_stride), k, relu != 0, sa, sb, sx);
        da += (double)sa;
        db += (double)sb;
        dx += (double)sx;
        __syncwarp();
    }
    s_red[0][warp][lane] = da;
    s_red[1][warp][lane] = db;
    s_red[2][warp][lane] = dx;
    __syncthreads();
    if (warp == 0) {
        double a = 0.0, b = 0.0, xs = 0.0;
        for (int w = 0; w < kRowsWarps; ++w) { a += s_red[0][w][lane]; b += s_red[1][w][lane]; xs += s_red[2][w][lane]; }
        double *out = partial + (((long long)n * C + c) * kBwdMaxParts + blockIdx.y) * 3;
        out[0] = a;
        out[1] = b;
        out[2] = xs;
    }
}



// apply: a warp turns a 32-pixel x 32-channel tile of grad_y (128-bit loads along the channels of one pixel) through
// shared memory, then each lane (= one pixel) walks the channels: reads of x and writes of grad_x along the pixels
__global__ void __launch_bounds__(kRowsWarps * 32)
gn_bwd_rows_apply_kernel(const float *__restrict__ gy, long long row_stride, long long image_stride,
                         const float *__restrict__ x, const float *__restrict__ mean_rstd,
                         const float *__restrict__ gamma, const float *__restrict__ beta,
                         const float *__restrict__ cbias, const double *__restrict__ ab, float *__restrict__ gx, int C,
                         long long hw, int cpg, int relu) {
    // blockIdx.x = image * (C / 32) + channel block, blockIdx.y = pixel range
    __shared__ GnChan s_k[32];
    __shared__ float s_k1[32], s_ka[32], s_kb[32];
    __shared__ float s_tile[kRowsWarps][32 * 33];
    const int cblocks = C / 32, n = blockIdx.x / cblocks, c0 = (blockIdx.x % cblocks) * 32;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x < 32) {
        const int c = c0 + threadIdx.x;
        const long long ng = (long long)n * (C / cpg) + c / cpg;
        const GnChan k = gn_chan(mean_rstd, ng, gamma, beta, cbias, c);
        s_k[threadIdx.x] = k;
        gn_bwd_factors(k, __ldg(gamma + c), ab, ng, (double)cpg * (double)hw, s_k1[threadIdx.x], s_ka[threadIdx.x],
                       s_kb[threadIdx.x]);
    }
    __syncthreads();
    float *tile = s_tile[warp];
    const float *xin = x + ((long long)n * C + c0) * hw;
    float *gout = gx + ((long long)n * C + c0) * hw;
    const float *gin = gy + (long long)n * image_stride + c0;
    const int sub = lane >> 3, ch4 = (lane & 7) * 4;
    const long long first = ((long long)blockIdx.y * kRowsWarps + warp) * kRowsTilesPerWarp;
    for (int t = 0; t < kRowsTilesPerWarp; ++t) {
        const long long p0 = (first + t) * 32;
        if (p0 >= hw) break;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int pix = i * 4 + sub;
            const float4 g = p0 + pix < hw ? ldg_stream_f4(reinterpret_cast<const float4 *>(gin + (p0 + pix) * row_stride + ch4))
                                           : make_float4(0.f, 0.f, 0.f, 0.f);
            tile[(ch4 + 0) * 33 + pix] = g.x;
            tile[(ch4 + 1) * 33 + pix] = g.y;
            tile[(ch4 + 2) * 33 + pix] = g.z;
            tile[(ch4 + 3) * 33 + pix] = g.w;
        }
        __syncwarp();
        const long long p = p0 + lane;
        if (p < hw) {
#pragma unroll 8
            for (int j = 0; j < 32; ++j) {
                const float v = ldg_stream_f1(xin + (long long)j * hw + p);
                gout[(long long)j * hw + p] = gn_bwd_dx(v, tile[j * 33 + lane], s_k[j], relu != 0, s_k1[j], s_ka[j], s_kb[j]);
            }
        }
        __syncwarp();
    }
}

// the same for a 16-bit x and grad_x: a copy of the fp32 source (DESIGN.md 11.3)
template <typename V>
__global__ void __launch_bounds__(kRowsWarps * 32)
gn_bwd_rows_apply_mixed_kernel(const float *__restrict__ gy, long long row_stride, long long image_stride,
                               const V *__restrict__ x, const float *__restrict__ mean_rstd,
                               const float *__restrict__ gamma, const float *__restrict__ beta,
                               const float *__restrict__ cbias, const double *__restrict__ ab, V *__restrict__ gx,
                               int C, long long hw, int cpg, int relu) {
    // blockIdx.x = image * (C / 32) + channel block, blockIdx.y = pixel range
    __shared__ GnChan s_k[32];
    __shared__ float s_k1[32], s_ka[32], s_kb[32];
    __shared__ float s_tile[kRowsWarps][32 * 33];
    const int cblocks = C / 32, n = blockIdx.x / cblocks, c0 = (blockIdx.x % cblocks) * 32;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x < 32) {
        const int c = c0 + threadIdx.x;
        const long long ng = (long long)n * (C / cpg) + c / cpg;
        const GnChan k = gn_chan(mean_rstd, ng, gamma, beta, cbias, c);
        s_k[threadIdx.x] = k;
        gn_bwd_factors(k, __ldg(gamma + c), ab, ng, (double)cpg * (double)hw, s_k1[threadIdx.x], s_ka[threadIdx.x],
                       s_kb[threadIdx.x]);
    }
    __syncthreads();
    float *tile = s_tile[warp];
    const V *xin = x + ((long long)n * C + c0) * hw;
    V *gout = gx + ((long long)n * C + c0) * hw;
    const float *gin = gy + (long long)n * image_stride + c0;
    const int sub = lane >> 3, ch4 = (lane & 7) * 4;
    const long long first = ((long long)blockIdx.y * kRowsWarps + warp) * kRowsTilesPerWarp;
    for (int t = 0; t < kRowsTilesPerWarp; ++t) {
        const long long p0 = (first + t) * 32;
        if (p0 >= hw) break;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int pix = i * 4 + sub;
            const float4 g = p0 + pix < hw ? ldg_stream_f4(reinterpret_cast<const float4 *>(gin + (p0 + pix) * row_stride + ch4))
                                           : make_float4(0.f, 0.f, 0.f, 0.f);
            tile[(ch4 + 0) * 33 + pix] = g.x;
            tile[(ch4 + 1) * 33 + pix] = g.y;
            tile[(ch4 + 2) * 33 + pix] = g.z;
            tile[(ch4 + 3) * 33 + pix] = g.w;
        }
        __syncwarp();
        const long long p = p0 + lane;
        if (p < hw) {
#pragma unroll 8
            for (int j = 0; j < 32; ++j) {
                const float v = ldg_stream_one<V>(xin + (long long)j * hw + p);
                gout[(long long)j * hw + p] =
                    narrow<V>(gn_bwd_dx(v, tile[j * 33 + lane], s_k[j], relu != 0, s_k1[j], s_ka[j], s_kb[j]));
            }
        }
        __syncwarp();
    }
}



// workspace (doubles): reduce-pass slots [N*C][kBwdMaxParts][3], per-plane sums [N*C][3], per-group sums [N*C][2]
// (groups <= C)
struct GnBwdWs {
    double *partial, *abx, *ab;
    GnBwdWs(double *w, long long planes)
        : partial(w), abx(w + planes * kBwdMaxParts * 3), ab(w + planes * (kBwdMaxParts * 3 + 3)) {}
};

}  // namespace

long long group_norm_bwd_workspace_doubles(int N, int C) { return (long long)N * C * (kBwdMaxParts * 3 + 3 + 2); }

// G: type of grad_y (float or V), V: of x and grad_x (float: the fp32 kernels; 16-bit: the mixed ones)
template <typename G, typename V>
cudaError_t launch_group_norm_bwd(const G *gy, const V *x, const float *cbias, const float *gamma,
                                  const float *beta, const float *mean_rstd, V *gx, float *ggamma, float *gbeta,
                                  float *gcbias, float *gup, int N, int C, int H, int W, int groups, int relu, int uh,
                                  int uw, double *workspace, cudaStream_t stream, bool *handled) {
    *handled = false;
    if (!gn_nchw_ok(N, C, H, W, groups, gup != nullptr, amap(x) | amap(gy) | amap(gx)) ||
        (gup != nullptr && (uh <= 0 || uw <= 0 || (long long)uh * uw > 0x7fffffffLL)))
        return cudaSuccess;
    *handled = true;
    const int cpg = C / groups;
    const long long hw = (long long)H * W, hw4 = hw >> 2;
    const GnBwdWs ws(workspace, (long long)N * C);
    int parts = (int)((hw4 + 4095) / 4096);
    parts = parts < 1 ? 1 : parts > kBwdMaxParts ? kBwdMaxParts : parts;
    const dim3 rgrid((unsigned)(N * C), (unsigned)parts);
    if constexpr (is16<V>) {
        if (relu) gn_bwd_reduce_mixed_kernel<G, V, true><<<rgrid, kBwdThreads, 0, stream>>>(gy, x, mean_rstd, gamma, beta, cbias, ws.partial, C, cpg, hw4);
        else gn_bwd_reduce_mixed_kernel<G, V, false><<<rgrid, kBwdThreads, 0, stream>>>(gy, x, mean_rstd, gamma, beta, cbias, ws.partial, C, cpg, hw4);
    } else {
        if (relu) gn_bwd_reduce_kernel<true><<<rgrid, kBwdThreads, 0, stream>>>(gy, x, mean_rstd, gamma, beta, cbias, ws.partial, C, cpg, hw4);
        else gn_bwd_reduce_kernel<false><<<rgrid, kBwdThreads, 0, stream>>>(gy, x, mean_rstd, gamma, beta, cbias, ws.partial, C, cpg, hw4);
    }
    note_launch();
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    gn_bwd_finalize_kernel<<<groups, kBwdThreads, 0, stream>>>(ws.partial, parts, gamma, mean_rstd, N, C, cpg, hw,
                                                               ws.abx, ws.ab, ggamma, gbeta, gcbias);
    note_launch();
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    int aparts = (int)((hw4 + 8191) / 8192);
    aparts = aparts < 1 ? 1 : aparts > 64 ? 64 : aparts;
    const dim3 agrid((unsigned)(N * C), (unsigned)aparts);
    if constexpr (is16<V>) {
        if (relu) gn_bwd_apply_mixed_kernel<G, V, true><<<agrid, kBwdThreads, 0, stream>>>(gy, x, mean_rstd, gamma, beta, cbias, ws.ab, gx, C, cpg, hw4);
        else gn_bwd_apply_mixed_kernel<G, V, false><<<agrid, kBwdThreads, 0, stream>>>(gy, x, mean_rstd, gamma, beta, cbias, ws.ab, gx, C, cpg, hw4);
    } else {
        if (relu) gn_bwd_apply_kernel<true><<<agrid, kBwdThreads, 0, stream>>>(gy, x, mean_rstd, gamma, beta, cbias, ws.ab, gx, C, cpg, hw4);
        else gn_bwd_apply_kernel<false><<<agrid, kBwdThreads, 0, stream>>>(gy, x, mean_rstd, gamma, beta, cbias, ws.ab, gx, C, cpg, hw4);
    }
    note_launch();
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    if (gup != nullptr) {
        const long long src = (long long)uh * uw;
        long long uparts = (src + 4 * kBwdThreads - 1) / (4 * kBwdThreads);
        uparts = uparts < 1 ? 1 : uparts > 64 ? 64 : uparts;
        const dim3 ugrid((unsigned)(N * C), (unsigned)uparts);
        if constexpr (is16<G>)
            gn_bwd_up_mixed_kernel<G><<<ugrid, kBwdThreads, 0, stream>>>(gy, gup, H, W, uh, uw, (float)uh / (float)H,
                                                                        (float)uw / (float)W);
        else
            gn_bwd_up_kernel<<<ugrid, kBwdThreads, 0, stream>>>(gy, gup, H, W, uh, uw, (float)uh / (float)H,
                                                                (float)uw / (float)W);
        note_launch();
        e = cudaGetLastError();
    }
    return e;
}

// fp32 grad_y rows; V: type of x and grad_x
template <typename V>
cudaError_t launch_group_norm_rows_bwd(const float *gy, long long row_stride, long long image_stride, const V *x,
                                       const float *cbias, const float *gamma, const float *beta,
                                       const float *mean_rstd, V *gx, float *ggamma, float *gbeta, float *gcbias,
                                       int N, int C, long long hw, int groups, int relu, double *workspace,
                                       cudaStream_t stream, bool *handled) {
    *handled = false;
    if (!gn_rows_ok(N, C, hw, groups, row_stride, image_stride, amap(x) | amap(gy) | amap(gx))) return cudaSuccess;
    *handled = true;
    const int cpg = C / groups;
    const GnBwdWs ws(workspace, (long long)N * C);
    long long parts = (hw + 32LL * kRowsWarps - 1) / (32LL * kRowsWarps);
    parts = parts > kBwdMaxParts ? kBwdMaxParts : parts;
    const unsigned cblocks = (unsigned)(N * (C / 32));
    if constexpr (is16<V>)
        gn_bwd_rows_reduce_mixed_kernel<V><<<dim3(cblocks, (unsigned)parts), kRowsWarps * 32, 0, stream>>>(
            gy, row_stride, image_stride, x, mean_rstd, gamma, beta, cbias, ws.partial, C, hw, cpg, relu);
    else
        gn_bwd_rows_reduce_kernel<<<dim3(cblocks, (unsigned)parts), kRowsWarps * 32, 0, stream>>>(
            gy, row_stride, image_stride, x, mean_rstd, gamma, beta, cbias, ws.partial, C, hw, cpg, relu);
    note_launch();
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    gn_bwd_finalize_kernel<<<groups, kBwdThreads, 0, stream>>>(ws.partial, (int)parts, gamma, mean_rstd, N, C, cpg, hw,
                                                               ws.abx, ws.ab, ggamma, gbeta, gcbias);
    note_launch();
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    if constexpr (is16<V>)
        gn_bwd_rows_apply_mixed_kernel<V><<<dim3(cblocks, (unsigned)gn_rows_parts(hw)), kRowsWarps * 32, 0, stream>>>(
            gy, row_stride, image_stride, x, mean_rstd, gamma, beta, cbias, ws.ab, gx, C, hw, cpg, relu);
    else
        gn_bwd_rows_apply_kernel<<<dim3(cblocks, (unsigned)gn_rows_parts(hw)), kRowsWarps * 32, 0, stream>>>(
            gy, row_stride, image_stride, x, mean_rstd, gamma, beta, cbias, ws.ab, gx, C, hw, cpg, relu);
    note_launch();
    return cudaGetLastError();
}

#define GN_BWD_INSTANTIATE(G, V)                                                                                       \
    template cudaError_t launch_group_norm_bwd<G, V>(const G *, const V *, const float *, const float *,                \
                                                     const float *, const float *, V *, float *, float *, float *,      \
                                                     float *, int, int, int, int, int, int, int, int, double *,         \
                                                     cudaStream_t, bool *);
GN_BWD_INSTANTIATE(float, float)
GN_BWD_INSTANTIATE(float, __nv_bfloat16)
GN_BWD_INSTANTIATE(__nv_bfloat16, __nv_bfloat16)
GN_BWD_INSTANTIATE(float, __half)
GN_BWD_INSTANTIATE(__half, __half)
#undef GN_BWD_INSTANTIATE
#define GN_ROWS_BWD_INSTANTIATE(V)                                                                                     \
    template cudaError_t launch_group_norm_rows_bwd<V>(const float *, long long, long long, const V *, const float *,   \
                                                       const float *, const float *, const float *, V *, float *,       \
                                                       float *, float *, int, int, long long, int, int, double *,       \
                                                       cudaStream_t, bool *);
GN_ROWS_BWD_INSTANTIATE(float)
GN_ROWS_BWD_INSTANTIATE(__nv_bfloat16)
GN_ROWS_BWD_INSTANTIATE(__half)
#undef GN_ROWS_BWD_INSTANTIATE

// x[n, c, :, :] += bias[c] in place (the bias of a convolution run without one), 128-bit accesses (16-bit x: 64-bit
// accesses, the sum in fp32 and rounded once)
namespace {
template <typename V>
__device__ __forceinline__ void channel_bias_body(Chunk<V> *__restrict__ x, const float *__restrict__ bias, int C,
                                                  long long hw4) {
    const int plane = blockIdx.x;
    const float b = __ldg(bias + plane % C);
    const long long per = (hw4 + gridDim.y - 1) / gridDim.y;
    const long long beg = (long long)blockIdx.y * per, end = min(beg + per, hw4);
    Chunk<V> *p = x + (long long)plane * hw4;
    for (long long i = beg + threadIdx.x; i < end; i += 256) {
        float4 v = ldg_chunk<V>(p + i);
        v.x += b; v.y += b; v.z += b; v.w += b;
        st_chunk<V>(p + i, v);
    }
}

__global__ void __launch_bounds__(256)
channel_bias_kernel(float4 *__restrict__ x, const float *__restrict__ bias, int C, long long hw4) {
    channel_bias_body<float>(x, bias, C, hw4);
}

template <typename V>
__global__ void __launch_bounds__(256)
channel_bias_mixed_kernel(uint2 *__restrict__ x, const float *__restrict__ bias, int C, long long hw4) {
    channel_bias_body<V>(x, bias, C, hw4);
}
}  // namespace

template <typename V>
cudaError_t launch_channel_bias(V *x, const float *bias, int N, int C, long long hw, cudaStream_t stream,
                                bool *handled) {
    *handled = false;
    if ((hw & 3) || (long long)N * C > 0x7fffffffLL || amap(x)) return cudaSuccess;
    *handled = true;
    int parts = (int)((hw / 4 + 8191) / 8192);
    parts = parts < 1 ? 1 : parts > 64 ? 64 : parts;
    const dim3 grid((unsigned)(N * C), (unsigned)parts);
    if constexpr (is16<V>)
        channel_bias_mixed_kernel<V><<<grid, 256, 0, stream>>>(reinterpret_cast<uint2 *>(x), bias, C, hw >> 2);
    else
        channel_bias_kernel<<<grid, 256, 0, stream>>>(reinterpret_cast<float4 *>(x), bias, C, hw >> 2);
    note_launch();
    return cudaGetLastError();
}
template cudaError_t launch_channel_bias<float>(float *, const float *, int, int, long long, cudaStream_t, bool *);
template cudaError_t launch_channel_bias<__nv_bfloat16>(__nv_bfloat16 *, const float *, int, int, long long,
                                                        cudaStream_t, bool *);
template cudaError_t launch_channel_bias<__half>(__half *, const float *, int, int, long long, cudaStream_t, bool *);

}  // namespace msda
