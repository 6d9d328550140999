// msda_fwd.cu -- forward MSDA kernel for sm_100a, specialised for 32 channels per head
// (the pixel-decoder shape: d_model 256 / 8 heads); value rows in fp32, or bf16 / fp16
// with fp32 locations, weights and sums (the mixed-precision op).
//
// Replaces the reference's ms_deformable_im2col_gpu_kernel
// (ms_deform_im2col_cuda.cuh:242-304), which runs one thread per output element
// and recomputes every sampling point's geometry in all 32 lanes.
//
// Design (see DESIGN.md section 4):
//   * persistent CTAs walk work items = (image n, head m, group of 8*WARPS queries);
//     when the queries are laid out like the value pixels (encoder self-attention)
//     a group is a 2-D tile of one level, so neighbouring queries' bilinear
//     footprints overlap in L1;
//   * each warp owns 8 consecutive queries of the item.  Phase 1: the 8*L*P
//     sampling points are spread over the lanes (one point per lane per round):
//     load (x, y, weight), run decompose() once per point and write the four
//     corner records {offset, bilinear*attention weight} to shared memory, one
//     plane per corner (conflict-free 8-byte stores);
//   * phase 2, per query: lane = corner*8 + chunk.  One 128-bit shared load gives a
//     lane its corner's records of TWO points; per point it fetches 16 bytes of that
//     corner's 128-byte value row (one LDG.128; a warp instruction covers the four
//     corner rows of a point) and accumulates 4 channels;
//   * the four corner groups are summed with a 3-shuffle reduce-scatter that leaves
//     one output channel per lane: the store is a single coalesced 128-byte line.
//
// The kernel is bound by the L1TEX data pipe: one wavefront per 128-byte value row
// (48 per (query, head)) plus the shared-memory wavefronts of the records
// (profiles/); the record layout exists to keep the latter small.
#include "msda_common.cuh"

namespace msda {

// QPW = queries per warp per item: their records are resident in shared memory together, so
// a smaller QPW leaves more of the SM's 228 KB to L1 (the value rows)
template <int LP, int WARPS, int TILE_W, int QPW>
struct FwdCfg {
    static_assert(LP % 2 == 0, "points are consumed in pairs");
    static constexpr int kQPW = QPW;
    static constexpr int kGroup = WARPS * kQPW;           // queries per item
    static constexpr int kTileH = kGroup / TILE_W;
    static constexpr int kRounds = (kQPW * LP + 31) / 32; // phase-1 rounds
    static constexpr int kRecPerWarp = kQPW * LP;         // records per corner plane
    // plane stride in records: +2 (16 bytes) so the four corner planes start 4 banks apart and the
    // 4-address LDS.128 of phase 2 is conflict-free (an unpadded stride is a multiple of 128 bytes)
    static constexpr int kPlane = kRecPerWarp + 2;
    static constexpr size_t kSmem = (size_t)WARPS * 4 * kPlane * sizeof(uint2);
    static_assert(TILE_W % QPW == 0 && kGroup % TILE_W == 0, "tile shape");
};

// V: element type of value / out (float, or 16-bit: a lane's chunk is then 8 bytes of a 64-byte row,
// loaded as LDG.64 and widened to fp32; the sums are fp32 and only the output store rounds).  FUSED with 16-bit V:
// the raw offsets / logits are of type V too (ProducerT), widened as they are loaded
// The body of both forward kernels.  STRIDED (phase1_records): the row strides / tables of `pr` may be set.  The
// shared memory is the kernel's.
template <typename V, int LP, int WARPS, int TILE_W, int QPW, bool FUSED, bool STRIDED>
__device__ __forceinline__ void fwd_d32_items(const V *__restrict__ value, const int64_t *__restrict__ shapes,
                                              const int64_t *__restrict__ lstart, const float *__restrict__ loc_arg,
                                              const float *__restrict__ attw_arg, const Producers pr, const Dims d,
                                              const int want_spatial, V *__restrict__ out, unsigned char *smem_raw,
                                              LevelTable &lt) {
    using Cfg = FwdCfg<LP, WARPS, TILE_W, QPW>;
    // the raw tensors are passed as float pointers whatever their type, so that the fp32 kernels keep their names
    using PT = ProducerT<V, FUSED>;
    const PT *__restrict__ loc = reinterpret_cast<const PT *>(loc_arg);
    const PT *__restrict__ attw = reinterpret_cast<const PT *>(attw_arg);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int corner = lane >> 3, chunk = lane & 7;
    // corner plane k of this warp: rec + k * kPlane, indexed by (query slot * LP + point)
    uint2 *rec = reinterpret_cast<uint2 *>(smem_raw) + (size_t)warp * 4 * Cfg::kPlane;

    fill_level_table(lt, shapes, lstart, d.L, d.P, d.S, d.Lq, Cfg::kGroup, Cfg::kTileH, TILE_W,
                     want_spatial);
    __syncthreads();

    const int M = d.M;
    const long long items = (long long)d.N * M * lt.groups;
    const uint32_t pix_stride = (uint32_t)M * 8u;          // float4 units per pixel

    for (long long item = blockIdx.x; item < items; item += gridDim.x) {
        const int m = (int)(item % M);
        const long long rest = item / M;
        const int g = (int)(rest % lt.groups);
        const long long n = rest / lt.groups;
        int q0, cnt;
        warp_queries(lt, d.L, g, warp, Cfg::kGroup, Cfg::kTileH, TILE_W, d.Lq, Cfg::kQPW, q0, cnt);

        // ---- phase 1: one sampling point per lane per round -> records ----
        phase1_records<FUSED, LP, Cfg::kQPW, Cfg::kPlane, false, PT, STRIDED>(lt, rec, nullptr, loc, attw, pr, n, q0, cnt, m,
                                                                 M, d.Lq, d.L, pix_stride, (uint32_t)d.S * pix_stride, lane);
        __syncwarp();

        // ---- phase 2: gather + weighted reduction, one query at a time ----
        const V *vb = value + (n * (long long)d.S * M * 8 + chunk) * 4;
        const uint4 *plane = reinterpret_cast<const uint4 *>(rec + corner * Cfg::kPlane);
        for (int qi = 0; qi < cnt; ++qi) {
            const uint4 *rq = plane + qi * (LP / 2);
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int sp2 = 0; sp2 < LP / 2; ++sp2) {
                const uint4 e = lds_u4(rq + sp2);           // this corner's records of 2 points
                if (e.x != kNoCorner) {
                    const float4 v = ldg_keep_v4(vb, e.x);
                    const float w = __uint_as_float(e.y);
                    acc.x = fmaf(w, v.x, acc.x);
                    acc.y = fmaf(w, v.y, acc.y);
                    acc.z = fmaf(w, v.z, acc.z);
                    acc.w = fmaf(w, v.w, acc.w);
                }
                if (e.z != kNoCorner) {
                    const float4 v = ldg_keep_v4(vb, e.z);
                    const float w = __uint_as_float(e.w);
                    acc.x = fmaf(w, v.x, acc.x);
                    acc.y = fmaf(w, v.y, acc.y);
                    acc.z = fmaf(w, v.z, acc.z);
                    acc.w = fmaf(w, v.w, acc.w);
                }
            }
            // sum the 4 corner groups (lane bits 3 and 4); lane ends with channel 4*chunk+corner
            const bool up16 = lane & 16, up8 = lane & 8;
            float a0 = up16 ? acc.z : acc.x, a1 = up16 ? acc.w : acc.y;
            const float s0 = up16 ? acc.x : acc.z, s1 = up16 ? acc.y : acc.w;
            a0 += __shfl_xor_sync(kFullMask, s0, 16);
            a1 += __shfl_xor_sync(kFullMask, s1, 16);
            const float keep = up8 ? a1 : a0, send = up8 ? a0 : a1;
            const float res = keep + __shfl_xor_sync(kFullMask, send, 8);
            V *o = out + ((n * d.Lq + q0 + qi) * M + m) * 32LL + chunk * 4 + corner;
            stg_stream_v1(o, res);
        }
        __syncwarp();   // records are overwritten by the next item
    }
}

template <typename V, int LP, int WARPS, int TILE_W, int MIN_CTAS, int QPW, bool FUSED>
__global__ void __launch_bounds__(WARPS * 32, MIN_CTAS)
msda_fwd_d32_kernel(const V *__restrict__ value, const int64_t *__restrict__ shapes,
                    const int64_t *__restrict__ lstart, const float *__restrict__ loc_arg,
                    const float *__restrict__ attw_arg, const Producers pr, const Dims d,
                    const int want_spatial, V *__restrict__ out) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ LevelTable lt;
    fwd_d32_items<V, LP, WARPS, TILE_W, QPW, FUSED, FUSED && !is16<V>>(value, shapes, lstart, loc_arg, attw_arg, pr, d,
                                                                      want_spatial, out, smem_raw, lt);
}

// the mixed-precision fused forward with row strides and / or per-query tables (16-bit V, raw 16-bit offsets / logits
// in rows of a [rows, 3*M*L*P] projection output, fp32 tables)
template <typename V, int LP, int WARPS, int TILE_W, int MIN_CTAS, int QPW>
__global__ void __launch_bounds__(WARPS * 32, MIN_CTAS)
msda_fwd_d32_strided_kernel(const V *__restrict__ value, const int64_t *__restrict__ shapes,
                            const int64_t *__restrict__ lstart, const float *__restrict__ loc_arg,
                            const float *__restrict__ attw_arg, const Producers pr, const Dims d,
                            const int want_spatial, V *__restrict__ out) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ LevelTable lt;
    fwd_d32_items<V, LP, WARPS, TILE_W, QPW, true, true>(value, shapes, lstart, loc_arg, attw_arg, pr, d, want_spatial,
                                                         out, smem_raw, lt);
}

// ---------------------------------------------------------------------------
// host side: launch_fwd_d32() serves the plain op and the fused producers (Producers::ref set),
// the latter in the default CTA shape only
// ---------------------------------------------------------------------------
// STRIDED: the 16-bit strided kernel (FUSED, 16-bit V)
template <typename V, int LP, int WARPS, int TILE_W, int MIN_CTAS, int QPW, bool FUSED, bool STRIDED = false>
static cudaError_t launch_fwd_cfg(const V *value, const int64_t *shapes, const int64_t *lstart,
                                  const ProducerT<V, FUSED> *loc, const ProducerT<V, FUSED> *attw, const Producers &pr,
                                  const Dims &d, V *out, cudaStream_t stream) {
    using Cfg = FwdCfg<LP, WARPS, TILE_W, QPW>;
    constexpr auto kern = [] {       // (only the kernel that is launched is instantiated)
        if constexpr (STRIDED) return msda_fwd_d32_strided_kernel<V, LP, WARPS, TILE_W, MIN_CTAS, QPW>;
        else return msda_fwd_d32_kernel<V, LP, WARPS, TILE_W, MIN_CTAS, QPW, FUSED>;
    }();
    cudaError_t e;
    const int blocks = persistent_blocks<kern>(WARPS * 32, Cfg::kSmem, d, &e);
    if (blocks == 0) return e;
    const int want_spatial = option_value(OPT_TILE_ORDER) != 1;
    kern<<<blocks, WARPS * 32, Cfg::kSmem, stream>>>(value, shapes, lstart, reinterpret_cast<const float *>(loc),
                                                     reinterpret_cast<const float *>(attw), pr, d, want_spatial, out);
    note_launch();
    return cudaGetLastError();
}

template <typename V, typename P, int LP>
static cudaError_t launch_fwd_lp(const V *value, const int64_t *shapes, const int64_t *lstart,
                                 const P *loc, const P *attw, const Producers &pr, const Dims &d,
                                 V *out, cudaStream_t stream) {
    // variant = (warps, query tile width, min CTAs per SM -> register budget, queries per warp)
#define MSDA_FWD(W, TW, C, Q, F) launch_fwd_cfg<V, LP, W, TW, C, Q, F>(value, shapes, lstart, loc, attw, pr, d, out, stream)
    if constexpr (is16<P>) {                                   // 16-bit fused producers: the default shape only
        if (pr.off_qstride != 0 || pr.off_table != nullptr)
            return launch_fwd_cfg<V, LP, 16, 16, 2, 8, true, true>(value, shapes, lstart, loc, attw, pr, d, out, stream);
        return MSDA_FWD(16, 16, 2, 8, true);
    } else if constexpr (is16<V>) {
        return MSDA_FWD(16, 16, 2, 8, false);                     // 16-bit plain: the default shape only
    } else {
    if (pr.ref != nullptr) return MSDA_FWD(16, 16, 2, 8, true);   // fused producers: the default shape only
    switch (option_value(OPT_FWD_VARIANT)) {
        case 1: return MSDA_FWD(8, 8, 4, 8, false);     //  8 warps, tile  8x8
        case 3: return MSDA_FWD(32, 16, 1, 8, false);   // 32 warps, tile 16x16, one CTA per SM
        case 4: return MSDA_FWD(16, 8, 2, 8, false);    // 16 warps, tile 16x8
        case 5: return MSDA_FWD(16, 16, 2, 4, false);   // 16 warps, tile  4x16, 4 queries per warp (50 KB smem per SM)
        case 6: return MSDA_FWD(16, 8, 2, 4, false);    // 16 warps, tile  8x8,  4 queries per warp
        case 7: return MSDA_FWD(32, 16, 1, 4, false);   // 32 warps, tile  8x16, 4 queries per warp, one CTA per SM
        case 8: return MSDA_FWD(16, 16, 3, 4, false);   // 16 warps, tile  4x16, 48 warps per SM (40 regs)
        case 2:
        default: return MSDA_FWD(16, 16, 2, 8, false);  // 16 warps, tile  8x16, 8 queries per warp (98 KB smem per SM)
    }
    }
#undef MSDA_FWD
}

// pr.ref == nullptr: plain, `loc` / `attw` are the sampling locations and attention weights.  Otherwise fused
// producers (SURVEY 8f.1): `loc` = raw sampling offsets, `attw` = raw attention logits, `pr.ref` = reference
// points [N or 1, Lq, L, 2].  `handled` = false: the problem is outside d32_applies() and nothing was launched.
// P: element type of `loc` / `attw` -- float, or V for the 16-bit fused producers (pr.ref set).
template <typename V, typename P>
cudaError_t launch_fwd_d32(const V *value, const int64_t *shapes, const int64_t *lstart, const P *loc,
                           const P *attw, const Producers &pr, const Dims &d, V *out, cudaStream_t stream,
                           bool *handled) {
    *handled = d32_applies(d);
    if (!*handled) return cudaSuccess;
    switch (d.L * d.P) {       // 4, 8, 12 or 16 (d32_applies)
        case 4: return launch_fwd_lp<V, P, 4>(value, shapes, lstart, loc, attw, pr, d, out, stream);
        case 8: return launch_fwd_lp<V, P, 8>(value, shapes, lstart, loc, attw, pr, d, out, stream);
        case 12: return launch_fwd_lp<V, P, 12>(value, shapes, lstart, loc, attw, pr, d, out, stream);
        default: return launch_fwd_lp<V, P, 16>(value, shapes, lstart, loc, attw, pr, d, out, stream);
    }
}

#define MSDA_FWD_D32(V, P)                                                                                         \
    template cudaError_t launch_fwd_d32<V, P>(const V *, const int64_t *, const int64_t *, const P *, const P *,  \
                                              const Producers &, const Dims &, V *, cudaStream_t, bool *);
MSDA_FWD_D32(float, float)
MSDA_FWD_D32(__nv_bfloat16, float)
MSDA_FWD_D32(__half, float)
MSDA_FWD_D32(__nv_bfloat16, __nv_bfloat16)
MSDA_FWD_D32(__half, __half)
#undef MSDA_FWD_D32

}  // namespace msda
