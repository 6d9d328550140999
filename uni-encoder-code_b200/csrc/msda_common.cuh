// msda_common.cuh -- shared device code for the sm_100a multi-scale deformable
// attention (MSDA) kernels.
//
// Nothing here is derived from the reference's CUDA sources; the arithmetic that
// must agree with them is cited by file:line (relative to
// /root/reference/model/modeling/pixel_decoder/ops/src/cuda/) next to the code.
#pragma once

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <atomic>
#include <cstring>
#include <type_traits>
#ifdef MSDA_CHECK_BOUNDS
#include <cassert>     // `make checked`: every corner offset is asserted to lie inside its image
#endif

namespace msda {

constexpr unsigned kFullMask = 0xffffffffu;
constexpr int kMaxLevels = 16;           // == MSDA_MAX_LEVELS in include/msda_b200.h
constexpr int kMaxSamples = 64;          // L*P bound for the shared sample->level table
constexpr int kMaxDevices = 64;          // per-device launch-attribute caches; higher ordinals are refused
constexpr uint32_t kNoCorner = 0xffffffffu;  // record marker: corner outside the level

// ---------------------------------------------------------------------------
// explicitly rounded helpers: the coordinate arithmetic below must not depend on the
// compiler's contraction choices
// ---------------------------------------------------------------------------
__device__ __forceinline__ float fma_rn(float a, float b, float c) { return __fmaf_rn(a, b, c); }
__device__ __forceinline__ double fma_rn(double a, double b, double c) { return __fma_rn(a, b, c); }
__device__ __forceinline__ float sub_rn(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ double sub_rn(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ int floor_to_int(float a) { return __float2int_rd(a); }
__device__ __forceinline__ int floor_to_int(double a) { return __double2int_rd(a); }

// ---------------------------------------------------------------------------
// Geometry of one sampling point.  This single function carries all the integer
// work that the parity tests pin bit-exactly (through msda_b200_debug_indices_f32):
//   pixel coordinate  x = fma(loc_x, W, -0.5), y = fma(loc_y, H, -0.5): ONE rounding.
//                     The source reads `loc * size - 0.5` (cuh:290-291); nvcc with the
//                     reference's build flags (default -fmad=true, ops/setup.py:44-49) folds the
//                     double literal and contracts it to a single FFMA -- `FFMA R, R, R, -0.5`
//                     in the SASS of the reference op built for sm_100
//                     (baseline/build_reference_cuda.py) -- so this is what the reference's
//                     kernels compute, and what we reproduce bit for bit
//   point valid       y > -1 && x > -1 && y < H && x < W         (cuh:293)
//   h_low, w_low      floor                                      (cuh:43-44)
//   lh, lw            fractional parts                           (cuh:48-49)
//   corner k valid    0 <= h <= H-1 && 0 <= w <= W-1             (cuh:60-83)
//     k = 0:(h_low,w_low) 1:(h_low,w_high) 2:(h_high,w_low) 3:(h_high,w_high)
// ---------------------------------------------------------------------------
template <typename T>
struct Geom {
    int valid;
    int h_low, w_low;
    int cmask;
    T lh, lw;
};

template <typename T>
__device__ __forceinline__ Geom<T> decompose(T loc_x, T loc_y, int H, int W) {
    Geom<T> g;
    const T h_im = fma_rn(loc_y, (T)H, (T)-0.5);
    const T w_im = fma_rn(loc_x, (T)W, (T)-0.5);
    g.valid = (h_im > (T)-1) && (w_im > (T)-1) && (h_im < (T)H) && (w_im < (T)W);
    g.h_low = floor_to_int(h_im);   // cvt.rmi saturates; NaN -> 0, and then valid == 0
    g.w_low = floor_to_int(w_im);
    g.lh = sub_rn(h_im, (T)g.h_low);
    g.lw = sub_rn(w_im, (T)g.w_low);
    int mask = 0;
    if (g.valid) {
        const bool h0 = g.h_low >= 0, h1 = g.h_low + 1 <= H - 1;
        const bool w0 = g.w_low >= 0, w1 = g.w_low + 1 <= W - 1;
        mask = (h0 && w0 ? 1 : 0) | (h0 && w1 ? 2 : 0) | (h1 && w0 ? 4 : 0) | (h1 && w1 ? 8 : 0);
    }
    g.cmask = mask;
    return g;
}

// ---------------------------------------------------------------------------
// Level table kept in shared memory by every kernel: the int64 device tensors
// spatial_shapes / level_start_index are read once per CTA instead of once per
// thread per level (the reference re-reads them inside its level loop, cuh:279-282).
// ---------------------------------------------------------------------------
struct LevelTable {
    int4 hws[kMaxLevels];             // {H, W, start, 0}: one 128-bit shared load per point in phase 1
    float2 rcp_wh[kMaxLevels];        // {RN(1/W), RN(1/H)} for div_by_size() (fused producers)
    int H[kMaxLevels];
    int W[kMaxLevels];
    int start[kMaxLevels];            // first pixel of the level inside one image
    int tiles_x[kMaxLevels];          // query tiles per row (spatial order only)
    int tile_begin[kMaxLevels + 1];   // prefix sum of tiles per level
    unsigned char level_of[kMaxSamples];  // sample index (l*P+p) -> l
    int spatial;                      // 1: queries are walked as 2-D tiles of the levels
    int groups;                       // query groups per (image, head)
};

// Fill the table.  Must be followed by __syncthreads().  `group` = queries per
// work item; tiles are tile_h x tile_w with tile_h*tile_w == group.
__device__ __forceinline__ void fill_level_table(LevelTable &lt, const int64_t *shapes,
                                                 const int64_t *lstart, int L, int P, int S,
                                                 int Lq, int group, int tile_h, int tile_w,
                                                 int want_spatial) {
    if (threadIdx.x == 0) {
        long long pix = 0;
        int tiles = 0;
        bool layout_ok = true;
        for (int l = 0; l < L; ++l) {
            const int H = (int)shapes[2 * l], W = (int)shapes[2 * l + 1];
            const long long st = lstart[l];
            lt.H[l] = H;
            lt.W[l] = W;
            lt.start[l] = (int)st;
            lt.hws[l] = make_int4(H, W, (int)st, 0);
            lt.rcp_wh[l] = make_float2(__frcp_rn((float)W), __frcp_rn((float)H));
            layout_ok = layout_ok && (st == pix) && H > 0 && W > 0;
            pix += (long long)H * W;
            lt.tiles_x[l] = (W + tile_w - 1) / tile_w;
            lt.tile_begin[l] = tiles;
            tiles += lt.tiles_x[l] * ((H + tile_h - 1) / tile_h);
        }
        lt.tile_begin[L] = tiles;
        // Spatial tiling only permutes the order in which queries are visited; it is
        // chosen when the queries are laid out like the value pixels (encoder
        // self-attention, msdeformattn.py:152-166), otherwise groups of consecutive
        // queries are used.  Either way every query is visited exactly once.
        const bool spatial = want_spatial && layout_ok && pix == (long long)S && Lq == S;
        lt.spatial = spatial ? 1 : 0;
        lt.groups = spatial ? tiles : (Lq + group - 1) / group;
    }
    for (int s = threadIdx.x; s < L * P && s < kMaxSamples; s += blockDim.x)
        lt.level_of[s] = (unsigned char)(s / P);
}

// First query and number of consecutive queries (0..qpw) handled by `warp` in
// query group `g` of an (image, head); qpw = queries per warp per item.
__device__ __forceinline__ void warp_queries(const LevelTable &lt, int L, int g, int warp,
                                             int group, int tile_h, int tile_w, int Lq, int qpw,
                                             int &q0, int &cnt) {
    if (lt.spatial) {
        int l = 0;
        while (l + 1 < L && g >= lt.tile_begin[l + 1]) ++l;
        const int t = g - lt.tile_begin[l];
        const int ty = t / lt.tiles_x[l], tx = t - ty * lt.tiles_x[l];
        const int per_row = tile_w / qpw;
        const int y = ty * tile_h + warp / per_row;
        const int x = tx * tile_w + (warp % per_row) * qpw;
        const int W = lt.W[l];
        cnt = (y < lt.H[l]) ? min(max(W - x, 0), qpw) : 0;
        q0 = lt.start[l] + y * W + x;
    } else {
        q0 = g * group + warp * qpw;
        cnt = min(max(Lq - q0, 0), qpw);
    }
}

// ---------------------------------------------------------------------------
// Per-point record shared by the 32-channel kernels: for each of the 4 bilinear
// corners {offset, weight}, offset in float4 units from the start of image n
// (pixel, head m, channel 0), weight = bilinear corner weight * attention weight.
// A corner outside the level -- or any corner of a point that fails the range test
// (cuh:293) -- gets {kNoCorner, 0}: it is neither read nor reduced into.
// ---------------------------------------------------------------------------
__device__ __forceinline__ void make_record(const Geom<float> &gm, float aw, uint32_t level_start,
                                            uint32_t W, uint32_t pix_stride, uint32_t head_off,
                                            uint32_t image_f4, uint4 &lo, uint4 &hi) {
    const float hh = 1.f - gm.lh, hw = 1.f - gm.lw;
    // modular uint32 arithmetic: h_low / w_low may be -1; contributing corners always land on
    // a true offset < 2^31 (checked on the host)
    const uint32_t base = (level_start + (uint32_t)gm.h_low * W + (uint32_t)gm.w_low) * pix_stride + head_off;
    const uint32_t row_stride = W * pix_stride;
    const int cm = gm.cmask;
    lo.x = (cm & 1) ? base : kNoCorner;
    lo.y = __float_as_uint((cm & 1) ? (hh * hw) * aw : 0.f);
    lo.z = (cm & 2) ? base + pix_stride : kNoCorner;
    lo.w = __float_as_uint((cm & 2) ? (hh * gm.lw) * aw : 0.f);
    hi.x = (cm & 4) ? base + row_stride : kNoCorner;
    hi.y = __float_as_uint((cm & 4) ? (gm.lh * hw) * aw : 0.f);
    hi.z = (cm & 8) ? base + row_stride + pix_stride : kNoCorner;
    hi.w = __float_as_uint((cm & 8) ? (gm.lh * gm.lw) * aw : 0.f);
#ifdef MSDA_CHECK_BOUNDS
    // a contributing corner's row [off, off + 8) float4 must lie inside image n (image_f4 = S*M*8)
    assert(!(cm & 1) || lo.x + 8u <= image_f4);
    assert(!(cm & 2) || lo.z + 8u <= image_f4);
    assert(!(cm & 4) || hi.x + 8u <= image_f4);
    assert(!(cm & 8) || hi.z + 8u <= image_f4);
    assert((lo.x == kNoCorner || (lo.x & 7u) == 0u) && (hi.z == kNoCorner || (hi.z & 7u) == 0u));
#else
    (void)image_f4;
#endif
}

// address = base + off16 * 16 in ONE instruction (IMAD.WIDE.U32); the compiler otherwise
// splits a 64-bit base that depends on the image index into several adds per access
template <typename T>
__device__ __forceinline__ T *at_off16(T *base, uint32_t off16) {
    unsigned long long r;
    asm("mad.wide.u32 %0, %1, 16, %2;" : "=l"(r) : "r"(off16), "l"((unsigned long long)base));
    return reinterpret_cast<T *>(r);
}

// one 128-bit shared load (the compiler otherwise splits it when half of it is only
// needed under a predicate); "memory": it reads records written earlier by other lanes
__device__ __forceinline__ uint4 lds_u4(const uint4 *p) {
    uint4 r;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "r"((uint32_t)__cvta_generic_to_shared(p))
                 : "memory");
    return r;
}

// ---------------------------------------------------------------------------
// cache-hinted global accesses
// ---------------------------------------------------------------------------
// value rows are re-used by neighbouring queries: keep them in L1
#ifndef MSDA_VALUE_LD
#define MSDA_VALUE_LD "ld.global.nc.v4.f32"   /* L1::evict_last measured: no change */
#endif
__device__ __forceinline__ float4 ldg_keep_f4(const float4 *p) {
    float4 r;
    asm(MSDA_VALUE_LD " {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
    return r;
}
// streamed once: do not allocate in L1
__device__ __forceinline__ float4 ldg_stream_f4(const float4 *p) {
    float4 r;
    asm("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ float2 ldg_stream_f2(const float2 *p) {
    float2 r;
    asm("ld.global.nc.L1::no_allocate.v2.f32 {%0,%1}, [%2];"
                 : "=f"(r.x), "=f"(r.y) : "l"(p));
    return r;
}
__device__ __forceinline__ float ldg_stream_f1(const float *p) {
    float r;
    asm("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(r) : "l"(p));
    return r;
}
__device__ __forceinline__ void stg_stream_f1(float *p, float v) {
    asm volatile("st.global.L1::no_allocate.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory");
}

// 128-bit vector reduction into global memory (sm_90+): one instruction adds four consecutive
// floats (SASS: REDG.E.ADD.F32x4).  Predicated forms used by the backward kernel: the validity test lives inside the asm block so
// that no C++ branch surrounds the access -- the loads stay freely schedulable (a batch of them is
// issued before the first use) and the reductions keep program order without fencing the loads.
__device__ __forceinline__ float4 ldg_keep_f4_if(const float4 *base, uint32_t off16) {
    float4 r;
    const float4 *p = at_off16(base, off16);
    asm("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %5, 0xffffffff;\n\t"
        "mov.f32 %0, 0f00000000;\n\tmov.f32 %1, 0f00000000;\n\tmov.f32 %2, 0f00000000;\n\t"
        "mov.f32 %3, 0f00000000;\n\t"
        "@p " MSDA_VALUE_LD " {%0,%1,%2,%3}, [%4];\n\t}"
        : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
        : "l"(p), "r"(off16));
    return r;
}
__device__ __forceinline__ void red_add_f4_if(float4 *base, uint32_t off16, float4 v) {
    float4 *p = at_off16(base, off16);
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %5, 0xffffffff;\n\t"
                 "@p red.global.add.v4.f32 [%0], {%1,%2,%3,%4};\n\t}"
                 ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "r"(off16)
                 : "memory");
}

// ---------------------------------------------------------------------------
// Element type of value / output / grad_output.  V = float, or one of the 16-bit types
// (__nv_bfloat16, __half) of the mixed-precision op: its rows are half as wide, but every
// sum stays fp32 -- loads widen to fp32, and only the final store of a result rounds to V.
// A "chunk" is 4 channels: the 16 (fp32) or 8 (16-bit) bytes a lane of the 32-channel
// kernels owns; the record offsets count chunks, so their meaning does not depend on V.
// ---------------------------------------------------------------------------
template <typename V>
constexpr bool is16 = sizeof(V) == 2;
template <typename V>
constexpr uint32_t kChunkBytes = 4 * sizeof(V);

template <typename T, typename V>
__device__ __forceinline__ T widen(V v) {
    if constexpr (std::is_same<V, __nv_bfloat16>::value) return (T)__bfloat162float(v);
    else if constexpr (std::is_same<V, __half>::value) return (T)__half2float(v);
    else return (T)v;
}
template <typename V, typename T>
__device__ __forceinline__ V narrow(T v) {
    if constexpr (std::is_same<V, __nv_bfloat16>::value) return __float2bfloat16_rn((float)v);
    else if constexpr (std::is_same<V, __half>::value) return __float2half_rn((float)v);   // overflow: +-inf
    else return (V)v;
}
// four 16-bit channels (8 bytes) -> fp32: a shift / mask for bf16, cvt for fp16
template <typename V>
__device__ __forceinline__ float4 widen4(uint2 u) {
    if constexpr (std::is_same<V, __nv_bfloat16>::value) {
        return make_float4(__uint_as_float(u.x << 16), __uint_as_float(u.x & 0xffff0000u),
                           __uint_as_float(u.y << 16), __uint_as_float(u.y & 0xffff0000u));
    } else {
        __half2 a, b;
        memcpy(&a, &u.x, 4);
        memcpy(&b, &u.y, 4);
        const float2 fa = __half22float2(a), fb = __half22float2(b);
        return make_float4(fa.x, fa.y, fb.x, fb.y);
    }
}
// address of chunk `off` from `base` in ONE instruction (see at_off16)
template <typename V>
__device__ __forceinline__ const V *at_chunk(const V *base, uint32_t off) {
    unsigned long long r;
    asm("mad.wide.u32 %0, %1, %2, %3;" : "=l"(r) : "r"(off), "n"(kChunkBytes<V>), "l"((unsigned long long)base));
    return reinterpret_cast<const V *>(r);
}
// a value chunk, kept in L1 (LDG.128 fp32, LDG.64 16-bit)
template <typename V>
__device__ __forceinline__ float4 ldg_keep_v4(const V *base, uint32_t off) {
    if constexpr (!is16<V>) {
        return ldg_keep_f4(reinterpret_cast<const float4 *>(at_chunk(base, off)));
    } else {
        uint2 u;
        asm("ld.global.nc.v2.u32 {%0,%1}, [%2];" : "=r"(u.x), "=r"(u.y) : "l"(at_chunk(base, off)));
        return widen4<V>(u);
    }
}
// the same, predicated on off != kNoCorner inside the asm (zeros otherwise), see ldg_keep_f4_if
template <typename V>
__device__ __forceinline__ float4 ldg_keep_v4_if(const V *base, uint32_t off) {
    if constexpr (!is16<V>) {
        return ldg_keep_f4_if(reinterpret_cast<const float4 *>(base), off);
    } else {
        uint2 u;
        asm("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %3, 0xffffffff;\n\t"
            "mov.b32 %0, 0;\n\tmov.b32 %1, 0;\n\t"
            "@p ld.global.nc.v2.u32 {%0,%1}, [%2];\n\t}"
            : "=r"(u.x), "=r"(u.y) : "l"(at_chunk(base, off)), "r"(off));
        return widen4<V>(u);
    }
}
// a chunk read once (grad_output rows)
template <typename V>
__device__ __forceinline__ float4 ldg_stream_v4(const V *p) {
    if constexpr (!is16<V>) {
        return ldg_stream_f4(reinterpret_cast<const float4 *>(p));
    } else {
        uint2 u;
        asm("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(u.x), "=r"(u.y) : "l"(p));
        return widen4<V>(u);
    }
}
// one result element, rounded to V
template <typename V>
__device__ __forceinline__ void stg_stream_v1(V *p, float v) {
    if constexpr (!is16<V>) {
        stg_stream_f1(reinterpret_cast<float *>(p), v);
    } else {
        const V h = narrow<V>(v);
        unsigned short bits;
        memcpy(&bits, &h, 2);
        asm volatile("st.global.L1::no_allocate.b16 [%0], %1;" ::"l"(p), "h"(bits) : "memory");
    }
}

// four consecutive results rounded to the 16-bit type H (round-to-nearest-even; fp16 overflow gives +-inf), one
// 8-byte store
template <typename H>
__device__ __forceinline__ void st_round4(H *p, float4 o) {
    const H a = narrow<H>(o.x), b = narrow<H>(o.y), c = narrow<H>(o.z), d = narrow<H>(o.w);
    unsigned short ba, bb, bc, bd;
    memcpy(&ba, &a, 2);
    memcpy(&bb, &b, 2);
    memcpy(&bc, &c, 2);
    memcpy(&bd, &d, 2);
    *reinterpret_cast<uint2 *>(p) = make_uint2((uint32_t)ba | ((uint32_t)bb << 16), (uint32_t)bc | ((uint32_t)bd << 16));
}

// ---------------------------------------------------------------------------
// Element type of the fused producers' raw tensors (sampling offsets, attention logits and their
// gradients): fp32, or -- in the mixed-precision fused op -- the value's 16-bit type, widened to fp32 on
// load and rounded once at the store.  The plain op's locations and weights are fp32 for every V.
// ---------------------------------------------------------------------------
template <typename V, bool FUSED>
using ProducerT = std::conditional_t<FUSED, V, float>;
// one (x, y) pair of offsets / locations: float2, or two 16-bit values in one 32-bit word
template <typename P>
using Pair = std::conditional_t<is16<P>, uint32_t, float2>;

template <typename P>
__device__ __forceinline__ float widen1(unsigned short bits) {
    if constexpr (std::is_same<P, __nv_bfloat16>::value) return __uint_as_float((uint32_t)bits << 16);
    else return __half2float(__ushort_as_half(bits));
}
template <typename P>
__device__ __forceinline__ float2 widen2(uint32_t u) {
    if constexpr (std::is_same<P, __nv_bfloat16>::value) {
        return make_float2(__uint_as_float(u << 16), __uint_as_float(u & 0xffff0000u));
    } else {
        __half2 h;
        memcpy(&h, &u, 4);
        return __half22float2(h);
    }
}
template <typename P>
__device__ __forceinline__ float2 widen_pair(Pair<P> v) {
    if constexpr (!is16<P>) return v;
    else return widen2<P>(v);
}
// a pair read once (LDG.64 fp32, one 4-byte load 16-bit), as loaded: 16-bit pairs take one register until widened
template <typename P>
__device__ __forceinline__ Pair<P> ldg_stream_pair_raw(const Pair<P> *p) {
    if constexpr (!is16<P>) {
        return ldg_stream_f2(p);
    } else {
        uint32_t u;
        asm("ld.global.nc.L1::no_allocate.b32 %0, [%1];" : "=r"(u) : "l"(p));
        return u;
    }
}
template <typename P>
__device__ __forceinline__ float2 ldg_stream_pair(const Pair<P> *p) {
    return widen_pair<P>(ldg_stream_pair_raw<P>(p));
}
// the same through the default cache path (the backward kernels' location probe)
template <typename P>
__device__ __forceinline__ float2 ld_pair(const Pair<P> *p) {
    if constexpr (!is16<P>) return *p;
    else return widen2<P>(*p);
}
// one element read once (a logit / attention weight)
template <typename P>
__device__ __forceinline__ float ldg_stream_one(const P *p) {
    if constexpr (!is16<P>) {
        return ldg_stream_f1(p);
    } else {
        unsigned short u;
        asm("ld.global.nc.L1::no_allocate.b16 %0, [%1];" : "=h"(u) : "l"(p));
        return widen1<P>(u);
    }
}
// one pair of results, each rounded to P (one 8-byte / 4-byte store)
template <typename P>
__device__ __forceinline__ void stg_stream_pair(Pair<P> *p, float x, float y) {
    if constexpr (!is16<P>) {
        asm volatile("st.global.L1::no_allocate.v2.f32 [%0], {%1,%2};" ::"l"(p), "f"(x), "f"(y) : "memory");
    } else {
        const P hx = narrow<P>(x), hy = narrow<P>(y);
        unsigned short bx, by;
        memcpy(&bx, &hx, 2);
        memcpy(&by, &hy, 2);
        asm volatile("st.global.L1::no_allocate.b32 [%0], %1;" ::"l"(p), "r"((uint32_t)bx | ((uint32_t)by << 16))
                     : "memory");
    }
}

// ---------------------------------------------------------------------------
// Warp reduce-scatter: n per-lane values are summed across the two lanes that
// differ in one lane-id bit; each lane keeps ceil(n/2) of the sums.  Repeating it
// over k bits sums across 2^k lanes with ~n shuffles in total instead of n*k.
// After a step, element i of a lane whose bit is `upper` holds the sum for input
// index i + upper*ceil(n/2) (absent if that is >= n).
// ---------------------------------------------------------------------------
template <int N>
__device__ __forceinline__ void rs_step(const float (&in)[N], float (&out)[(N + 1) / 2],
                                        bool upper, int lane_xor) {
    constexpr int H = (N + 1) / 2;
#pragma unroll
    for (int i = 0; i < H; ++i) {
        const float lo = in[i];
        const float hi = (i + H < N) ? in[i + H] : 0.f;
        const float keep = upper ? hi : lo;
        const float send = upper ? lo : hi;
        out[i] = keep + __shfl_xor_sync(kFullMask, send, lane_xor);
    }
}

// ---------------------------------------------------------------------------
// Phase 1 of the 32-channel kernels: the QPW*LP sampling points of a warp's queries are spread
// over the lanes (one point per lane per round); each lane produces its point's four corner
// records (one shared-memory plane per corner) and, for the backward kernel, the per-point
// coefficients {lh, lw, attention weight, level}.
//
// FUSED == false: (x, y) and the attention weight are read from sampling_locations /
//                 attention_weights, as in the reference op.
// FUSED == true : the producers of ops/modules/ms_deform_attn.py:105-112 are folded in:
//                 `loc`  = raw sampling_offsets  [N, Lq, M, L, P, 2]   (Linear output)
//                 `attw` = raw attention logits  [N, Lq, M, L*P]       (Linear output)
//                 `ref`  = reference points      [N or 1, Lq, L, 2]
//                 location = ref + offset / (W_l, H_l)  (IEEE division, then add: the same two
//                 roundings as the reference's tensor expression) and the weight is the softmax
//                 of the query-head's L*P logits (exchanged through the warp's record area).
// ---------------------------------------------------------------------------
// a / b, correctly rounded (== __fdiv_rn), for a level size b with rb = RN(1/b): one Newton
// correction of a * rb through the exact FMA residual (Markstein).  Exact whenever nothing
// under- or overflows -- checked against IEEE division for every size up to 5000 on 1.5e9
// random numerators -- so numerators outside [1e-18, 1e18] (and inf / nan) take the full division.
__device__ __forceinline__ float div_by_size(float a, float b, float rb) {
    const float q0 = a * rb;
    const float q = fmaf(fmaf(-q0, b, a), rb, q0);
    const float mag = fabsf(a);
    if (!(mag < 1e18f) || (mag < 1e-18f && a != 0.f)) return __fdiv_rn(a, b);
    return q;
}

struct Producers {
    const float *ref;          // FUSED only; the host launchers pick the plain kernels when it is null
    long long ref_bstride;     // elements between images in `ref` (0: shared by the batch)
    // FUSED forward only: floats between consecutive queries' rows of the raw offsets / logits (0: packed,
    // M*L*P*2 and M*L*P) -- lets both live in one [rows, M*L*P*3] projection output
    int off_qstride;
    int logit_qstride;
    // FUSED forward only: per-QUERY additive tables (same row strides, Lq rows, shared by the batch), or null:
    // the position-embedding part of the two query projections, (src + pos) W^T = src W^T + pos W^T
    const float *off_table;
    const float *logit_table;
};

// PT: element type of `loc` / `attw` (ProducerT: 16-bit only for the mixed-precision fused op).  STRIDED: the row
// strides and tables of Producers may be set -- every fp32 fused kernel, and the 16-bit strided forward, whose raw
// values are widened first and then get their fp32 table entries added
template <bool FUSED, int LP, int QPW, int PLANE, bool WITH_AUX, typename PT, bool STRIDED = FUSED && !is16<PT>>
__device__ __forceinline__ void phase1_records(const LevelTable &lt, uint2 *rec, float4 *aux,
                                               const PT *__restrict__ loc,
                                               const PT *__restrict__ attw, const Producers pr,
                                               long long n, int q0, int cnt, int m, int M, int Lq,
                                               int L, uint32_t pix_stride, uint32_t image_f4, int lane) {
    constexpr int kRounds = (QPW * LP + 31) / 32;
    constexpr bool kStrided = STRIDED;             // row strides / tables may be set
    constexpr bool kWidened = STRIDED && is16<PT>;  // 16-bit pairs widened as loaded (a table entry may be added)
    // as loaded (16-bit: widened where used, one register per pair until then -- unless kWidened)
    std::conditional_t<kWidened, float2, Pair<PT>> xy[kRounds];
    float aw[kRounds];          // attention weight; FUSED: the raw logit until the softmax below
    float2 txy[FUSED ? kRounds : 1];   // FUSED with tables: the table entries, added once ALL loads are in flight
    float taw[FUSED ? kRounds : 1];
    const long long tab_li = kStrided ? n * Lq * (long long)((pr.off_qstride != 0 ? pr.off_qstride : M * LP * 2) >> 1) : 0;
    const long long tab_ai = kStrided ? n * Lq * (long long)(pr.logit_qstride != 0 ? pr.logit_qstride : M * LP) : 0;
#pragma unroll
    for (int r = 0; r < kRounds; ++r) {          // all global loads first
        const int s = r * 32 + lane;
        const int qi = s / LP, sp = s - qi * LP;
        xy[r] = {};
        aw[r] = 0.f;
        if (FUSED) {
            txy[r] = make_float2(0.f, 0.f);
            taw[r] = 0.f;
        }
        if (qi < cnt) {                           // also false for the padding lanes of the last round
            const long long qrow = (n * Lq + q0 + qi) * M + m;
            long long li = qrow * LP + sp, ai = li;
            if (kStrided && pr.off_qstride != 0) {
                const long long q = n * Lq + q0 + qi;
                li = q * (pr.off_qstride >> 1) + m * LP + sp;
                ai = q * pr.logit_qstride + m * LP + sp;
            }
            if constexpr (kWidened) xy[r] = ldg_stream_pair<PT>(reinterpret_cast<const Pair<PT> *>(loc) + li);
            else xy[r] = ldg_stream_pair_raw<PT>(reinterpret_cast<const Pair<PT> *>(loc) + li);
            aw[r] = ldg_stream_one<PT>(attw + ai);
            if (kStrided && pr.off_table != nullptr) {
                // the tables have Lq rows with the projections' row strides: entry = the projection's index
                // minus the image's n * Lq rows (tab_li / tab_ai below).  Reused by every image, but by one warp
                // per image: kept out of L1 (whose lines phase 2's value rows live on), served by L2
                txy[r] = ldg_stream_f2(reinterpret_cast<const float2 *>(pr.off_table) + (li - tab_li));
                taw[r] = ldg_stream_f1(pr.logit_table + (ai - tab_ai));
            }
        }
    }
    if constexpr (kStrided) {
        if (pr.off_table != nullptr) {
#pragma unroll
            for (int r = 0; r < kRounds; ++r) {
                xy[r].x += txy[r].x;
                xy[r].y += txy[r].y;
                aw[r] += taw[r];
            }
        }
    }
    if (FUSED) {
        // softmax over each (query, head) row's LP logits (mod.py:107-108).  The rows do not line up
        // with lanes (LP = 12), so the logits are exchanged through the warp's record area, which is
        // free until the records are written below: four lanes per query reduce its row to
        // {max, sum of exp}, then every lane normalises its own logit.
        static_assert(LP % 4 == 0 && (QPW * LP + 2 * QPW) * 4 <= 4 * PLANE * 8, "softmax scratch");
        float *scr = reinterpret_cast<float *>(rec);
        float2 *stats = reinterpret_cast<float2 *>(scr + QPW * LP);
#pragma unroll
        for (int r = 0; r < kRounds; ++r) {
            const int s = r * 32 + lane;
            if (s < cnt * LP) scr[s] = aw[r];
        }
        __syncwarp();
        {   // four lanes per query, LP/4 logits each; max and sum combined over lane bits 0,1
            static_assert(QPW * 4 <= 32, "one warp reduces all rows at once");
            const int q = min(lane >> 2, QPW - 1);
            const float *part = scr + q * LP + (lane & 3) * (LP / 4);
            float v[LP / 4];
#pragma unroll
            for (int k = 0; k < LP / 4; ++k) v[k] = part[k];
            float mx = v[0];
#pragma unroll
            for (int k = 1; k < LP / 4; ++k) mx = fmaxf(mx, v[k]);
            mx = fmaxf(mx, __shfl_xor_sync(kFullMask, mx, 1));
            mx = fmaxf(mx, __shfl_xor_sync(kFullMask, mx, 2));
            float sum = 0.f;
#pragma unroll
            for (int k = 0; k < LP / 4; ++k) sum += expf(v[k] - mx);
            sum += __shfl_xor_sync(kFullMask, sum, 1);
            sum += __shfl_xor_sync(kFullMask, sum, 2);
            if ((lane & 3) == 0 && (lane >> 2) < cnt) stats[lane >> 2] = make_float2(mx, sum);
        }
        __syncwarp();
#pragma unroll
        for (int r = 0; r < kRounds; ++r) {
            const int s = r * 32 + lane;
            const int qi = s / LP;
            if (qi < cnt) {
                const float2 st = stats[qi];
                aw[r] = __fdiv_rn(expf(aw[r] - st.x), st.y);
            }
        }
        __syncwarp();                             // the scratch is overwritten by the records
    }
#pragma unroll
    for (int r = 0; r < kRounds; ++r) {
        const int s = r * 32 + lane;
        const int qi = s / LP, sp = s - qi * LP;
        if (qi < cnt) {
            const int l = lt.level_of[sp];
            const int4 lv = lt.hws[l];            // {H, W, start, -}
            float2 xyf;
            if constexpr (kWidened) xyf = xy[r];
            else xyf = widen_pair<PT>(xy[r]);
            float x = xyf.x, y = xyf.y;
            if (FUSED) {
                const long long rrow = n * pr.ref_bstride + ((long long)(q0 + qi) * L + l) * 2;
                const float2 rp = ldg_stream_f2(reinterpret_cast<const float2 *>(pr.ref + rrow));
                const float2 rc = lt.rcp_wh[l];
                x = rp.x + div_by_size(x, (float)lv.y, rc.x);   // mod.py:110-112: ref + off / (W, H)
                y = rp.y + div_by_size(y, (float)lv.x, rc.y);
            }
            const Geom<float> gm = decompose(x, y, lv.x, lv.y);
            uint4 lo, hi;   // {off0, w0, off1, w1}, {off2, w2, off3, w3}
            make_record(gm, aw[r], (uint32_t)lv.z, (uint32_t)lv.y, pix_stride, (uint32_t)m * 8u, image_f4, lo, hi);
            rec[0 * PLANE + s] = make_uint2(lo.x, lo.y);
            rec[1 * PLANE + s] = make_uint2(lo.z, lo.w);
            rec[2 * PLANE + s] = make_uint2(hi.x, hi.y);
            rec[3 * PLANE + s] = make_uint2(hi.z, hi.w);
            if (WITH_AUX) {
                // invalid point: every D_k is 0 (no corner is read), so any finite lh / lw give the
                // reference's zero location / weight gradients (cuh:370-372); its attention weight is
                // kept because the fused softmax backward needs it (-a_i * sum_j a_j g_j)
                aux[s] = make_float4(gm.valid ? gm.lh : 0.f, gm.valid ? gm.lw : 0.f, aw[r], __int_as_float(l));
            }
        }
    }
}

// ---------------------------------------------------------------------------
// Which backward kernel?  (encoder self-attention, Lq == S)
// Merging grad_value contributions inside the SM (msda_bwd_sorted.cu) pays when the sampling points
// stay near their query (the encoder: offsets of a few pixels, ms_deform_attn.py:71-77); with
// locations spread over the whole image nearly every record is a run of one and the per-row
// reduction kernel (msda_bwd.cu) is faster.  The host cannot look at the locations (no device
// read-back, CUDA-graph capturable), so BOTH kernels are launched and every CTA of both first runs
// this probe: kProbeSamples pseudo-random (image, query, head, point) samples, the same in every CTA
// and in both kernels, and the fraction of them that lands within the merge windows' margin of its
// query.  The verdict is therefore identical everywhere; the kernel it goes against returns at once.
// Must be called by all threads of the CTA, after fill_level_table() + __syncthreads().
// ---------------------------------------------------------------------------
constexpr int kProbeSamples = 512;      // one per thread of a 16-warp CTA: one round of loads (1024: + 2 us per backward)
constexpr float kProbeMarginPx = 8.f;     // kSortMargin - 1 (msda_bwd_sorted.cu)
enum { GATE_NONE = 0, GATE_RUN_IF_LOCAL = 1, GATE_RUN_IF_SPREAD = 2 };

// FUSED: `loc` holds the raw sampling offsets, which ARE the distance from the query's own position in
// pixels of the sampled level (location = ref + offset / (W, H), mod.py:110-112).
template <bool FUSED = false, typename PT = float>
__device__ __forceinline__ bool probe_points_stay_local(const LevelTable &lt, const PT *__restrict__ loc,
                                                        int N, int Lq, int M, int L, int P) {
    __shared__ int probe_in, probe_all;
    if (threadIdx.x == 0) { probe_in = 0; probe_all = 0; }
    __syncthreads();
    const int LP = L * P;
    int n_in = 0, n_all = 0;
    if (lt.spatial) {
        for (int i = threadIdx.x; i < kProbeSamples; i += blockDim.x) {
            uint32_t h = (uint32_t)i * 2654435761u + 12345u;      // which (image, query, head, point)
            h ^= h >> 15; h *= 2246822519u; h ^= h >> 13;
            const int n = (int)(h % (uint32_t)N);
            h = h * 1664525u + 1013904223u;
            const int q = (int)((h >> 4) % (uint32_t)Lq);
            h = h * 1664525u + 1013904223u;
            const int m = (int)((h >> 8) % (uint32_t)M), sp = (int)((h >> 16) % (uint32_t)LP);
            if (FUSED) {
                const float2 off = ld_pair<PT>(reinterpret_cast<const Pair<PT> *>(loc) + ((((long long)n * Lq + q) * M + m) * LP + sp));
                ++n_all;
                if (fabsf(off.x) <= kProbeMarginPx && fabsf(off.y) <= kProbeMarginPx) ++n_in;
                continue;
            }
            int lq = 0;
            while (lq + 1 < L && q >= lt.start[lq + 1]) ++lq;
            const int qy = (q - lt.start[lq]) / lt.W[lq], qx = (q - lt.start[lq]) - qy * lt.W[lq];
            const int l = sp / P;
            const float2 xy = reinterpret_cast<const float2 *>(loc)[(((long long)n * Lq + q) * M + m) * LP + sp];
            const float W = (float)lt.W[l], H = (float)lt.H[l];
            const float x = xy.x * W - 0.5f, y = xy.y * H - 0.5f;
            if (x > -1.f && y > -1.f && x < W && y < H) {         // the op's own range test (cuh:293)
                const float rx = ((float)qx + 0.5f) * (W / (float)lt.W[lq]) - 0.5f;
                const float ry = ((float)qy + 0.5f) * (H / (float)lt.H[lq]) - 0.5f;
                ++n_all;
                if (fabsf(x - rx) <= kProbeMarginPx && fabsf(y - ry) <= kProbeMarginPx) ++n_in;
            }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        n_in += __shfl_xor_sync(kFullMask, n_in, o);
        n_all += __shfl_xor_sync(kFullMask, n_all, o);
    }
    if ((threadIdx.x & 31) == 0 && n_all) { atomicAdd(&probe_in, n_in); atomicAdd(&probe_all, n_all); }
    __syncthreads();
    return probe_all > 0 && 4 * probe_in >= 3 * probe_all;       // >= 75 % near their query: merge
}

// ---------------------------------------------------------------------------
// launch bookkeeping shared by the translation units
// ---------------------------------------------------------------------------
struct Dims {
    int N, S, M, D, L, Lq, P;
};

// Deterministic backward (msda_det.cu): instead of reducing into grad_value, the backward kernels
// write one record per (sampling point, corner) into the fixed slot
//     ((((n*Lq + q)*M + m)*L + l)*P + p)*4 + corner
// key[slot] = destination grad_value row (n*S + pixel)*M + m, or `sentinel` (= N*S*M) for a corner that
// does not contribute; slot_id[slot] = slot (the values the stable sort carries); w[slot] = bilinear corner
// weight * attention weight (of the value type: float or double; 0 for the sentinel).
struct DetRecords {
    uint32_t *key;
    uint32_t *slot_id;
    void *w;
    uint32_t sentinel;
};
// the deterministic backward's workspace (msda_det.cu)
struct DetLayout {
    long long records;          // N*Lq*M*L*P*4
    uint32_t rows;              // N*S*M: grad_value rows, also the sentinel key
    int end_bit;                // bit width of `rows`
    size_t keys_a, keys_b, ids_a, ids_b, w, start, temp;   // byte offsets into the workspace
    size_t temp_bytes, total;
};
bool det_layout(const Dims &d, int value_bytes, DetLayout *out);
DetRecords det_records(void *ws, const DetLayout &l);
// V: element type of grad_output / grad_value; T: of the record weights and the sums (float for 16-bit V)
template <typename V, typename T>
cudaError_t launch_det_reduce(const DetLayout &l, void *ws, const V *grad_out, V *grad_value, const Dims &d,
                              cudaStream_t stream);

void note_launch();                   // increments the library launch counter
int sm_count();                       // SMs of the current device (cached)
int option_value(int which);          // tuning knobs, see msda_api.cu
enum { OPT_FWD_VARIANT = 0, OPT_BWD_VARIANT = 1, OPT_TILE_ORDER = 2, OPT_CTAS_PER_SM = 3,
       OPT_WHATIF_DROP_REDS = 4, OPT_LINEAR_VARIANT = 5, OPT_WHATIF_LINEAR = 6, OPT_WGRAD_CHUNK = 7,
       OPT_COUNT = 8 };
// The two what-if knobs make kernels skip work ON PURPOSE (wrong results, timing experiments for
// profiles/ only): they exist only in a library built with -DMSDA_PROFILE_KNOBS (`make profile`);
// in the shipped library they read as 0 and cannot be set.
#ifdef MSDA_PROFILE_KNOBS
inline int whatif_value(int which) { return option_value(which); }
#else
inline int whatif_value(int) { return 0; }
#endif
// Slot of the current device in the per-device launch-attribute caches, -1 with *err set when the
// device cannot be determined or its ordinal is beyond kMaxDevices (never aliased onto device 0).
inline int device_slot(cudaError_t *err) {
    int dev = 0;
    *err = cudaGetDevice(&dev);
    if (*err != cudaSuccess) return -1;
    if (dev < 0 || dev >= kMaxDevices) { *err = cudaErrorInvalidDevice; return -1; }
    return dev;
}

// Domain of the 32-channel kernels (msda_fwd.cu, msda_bwd.cu, msda_bwd_sorted.cu): D == 32, an instantiated
// point count L*P, and float4 offsets into an image of value / grad_value that fit in 31 bits.
inline bool d32_applies(const Dims &d) {
    const int lp = d.L * d.P;
    return d.D == 32 && (long long)d.S * d.M * 8 < 0x7fffffffLL && (lp == 4 || lp == 8 || lp == 12 || lp == 16);
}

// Grid of the persistent kernel `Kern`: as many CTAs as fit on an SM (capped by "ctas_per_sm") on every SM, but
// no more than N*M*Lq (every work item holds at least one query).  The opt-in shared-memory size is a per-device
// function attribute: it is set, and the occupancy queried, once per device and kernel instance; the values are
// immutable afterwards.  Returns 0 with *err set when a CUDA call fails.
template <auto Kern>
int persistent_blocks(int threads, size_t smem, const Dims &d, cudaError_t *err) {
    static std::atomic<int> ctas_per_sm_of[kMaxDevices];
    const int dev = device_slot(err);
    if (dev < 0) return 0;
    int per_sm = ctas_per_sm_of[dev].load(std::memory_order_acquire);
    if (per_sm == 0) {
        *err = cudaFuncSetAttribute(Kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (*err != cudaSuccess) return 0;
        int nb = 0;
        *err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, Kern, threads, smem);
        if (*err != cudaSuccess) return 0;
        per_sm = nb > 0 ? nb : 1;
        ctas_per_sm_of[dev].store(per_sm, std::memory_order_release);
    }
    const int cap = option_value(OPT_CTAS_PER_SM);
    if (cap > 0 && cap < per_sm) per_sm = cap;
    long long blocks = (long long)sm_count() * per_sm;
    const long long items_ub = (long long)d.N * d.M * d.Lq;
    if (blocks > items_ub) blocks = items_ub;
    return blocks < 1 ? 1 : (int)blocks;
}

}  // namespace msda
