// msda_bwd.cu -- backward MSDA kernel for sm_100a, 32 channels per head (fp32 value rows, or bf16 / fp16
// ones with fp32 locations, weights, sums and grad_value accumulation).
//
// Replaces the reference's col2im kernel that is hit at D = 32,
// ms_deformable_col2im_gpu_kernel_shm_blocksize_aware_reduce_v1<T,32>
// (ms_deform_im2col_cuda.cuh:306-408) and its bilinear helper (cuh:92-164):
// there every (query, head) is a 32-thread block that, per sampling point, issues
// 128 scalar atomicAdds, writes 3 partials per thread to shared memory and lets
// thread 0 add them up serially between two __syncthreads.
//
// Design (same work decomposition, phase 1 and record layout as msda_fwd.cu):
//   * the L*P points of a query are consumed in batches of BATCH record pairs: the 2*BATCH
//     value loads of a batch are issued before the first of them is used.  The shipped
//     BATCH is 1 (64 registers, 32 warps per SM): larger batches spill or halve the
//     occupancy and measured slower (profiles/r1_sweep.md);
//   * the corner validity test lives inside the asm of the load / reduction (@p ld / @p red),
//     so no C++ branch surrounds them;
//   * lane = corner*8 + chunk.  Per sampling point a lane loads 16 bytes of its
//     corner's value row, forms the partial dot product with its 4 grad_output
//     channels (d) and adds weight*grad_output to grad_value with ONE 128-bit
//     vector reduction (red.global.add.v4.f32) -- 4 warp-level REDG per point
//     row instead of 128 scalar ones, no shared-memory atomics (fp32 shared atomics
//     are CAS loops on sm_100a);
//   * grad_sampling_loc and grad_attn_weight are linear in the four per-corner dot
//     products D_k = sum_c v_k[c]*g[c].  The L*P partials d are kept in registers
//     and summed over the 8 lanes of each corner group with a reduce-scatter
//     (11 shuffles for 12 points), multiplied by the per-corner coefficients, and
//     summed over the 4 corner groups with a second reduce-scatter (5 shuffles):
//     16 shuffles and no barrier per (query, head) instead of 24 barriers and a
//     serial 32-term sum per point.  The summation order is fixed, so these two
//     outputs are deterministic; only grad_value depends on reduction order.
#include "msda_common.cuh"

namespace msda {

// QPW = queries per warp per item: their records are resident in shared memory together, so
// a smaller QPW leaves more of the SM's 228 KB to L1 (the value rows)
template <int LP, int WARPS, int TILE_W, int QPW>
struct BwdCfg {
    static_assert(LP % 2 == 0, "points are consumed in pairs");
    static constexpr int kPairs = LP / 2;            // record pairs per query
    static constexpr int kQPW = QPW;
    static constexpr int kGroup = WARPS * kQPW;
    static constexpr int kTileH = kGroup / TILE_W;
    static constexpr int kRounds = (kQPW * LP + 31) / 32;
    static constexpr int kRecPerWarp = kQPW * LP;
    static constexpr int kPlane = kRecPerWarp + 2;   // padded corner-plane stride, see msda_fwd.cu
    // per warp: 4 corner planes of {offset, weight} + one {lh, lw, attention weight, level} per point
    static constexpr size_t kRecBytes = (size_t)WARPS * 4 * kPlane * sizeof(uint2);
    static constexpr size_t kSmem = kRecBytes + (size_t)WARPS * kRecPerWarp * sizeof(float4);
    // sizes along the two reduce-scatters
    static constexpr int kN1 = (LP + 1) / 2, kN2 = (kN1 + 1) / 2, kN3 = (kN2 + 1) / 2;  // per-lane D count
    static constexpr int kT0 = 3 * kN3, kT1 = (kT0 + 1) / 2, kT2 = (kT1 + 1) / 2;
};

// BATCH = record pairs whose 2*BATCH value loads are in flight together (register budget)
// RECORDS: deterministic mode (msda_det.cu) -- grad_value is not touched; each corner's {destination row,
// weight} goes to its fixed slot of `det` instead (chunk lane 0 of each corner group writes it)
// FUSED: `loc` / `attw` are the raw sampling offsets / attention logits and `grad_loc` / `grad_attw`
// receive the gradients with respect to THEM (offset gradient = location gradient / (W, H);
// softmax backward folded in), see phase1_records() in msda_common.cuh.
// V: element type of grad_out / value (16-bit: 8-byte lane loads widened to fp32); grad_value is fp32 either way --
// for 16-bit V the zero-filled accumulation buffer that msda_api.cu rounds into the 16-bit grad_value afterwards.
// FUSED with 16-bit V: the raw offsets / logits and their gradients are of type V too (ProducerT), widened as they
// are loaded and rounded once as they are stored
template <typename V, int LP, int WARPS, int TILE_W, int MIN_CTAS, int BATCH, int QPW, bool FUSED, bool RECORDS>
__global__ void __launch_bounds__(WARPS * 32, MIN_CTAS)
msda_bwd_d32_kernel(const V *__restrict__ grad_out, const V *__restrict__ value,
                    const int64_t *__restrict__ shapes, const int64_t *__restrict__ lstart,
                    const float *__restrict__ loc_arg, const float *__restrict__ attw_arg,
                    const Producers pr, const Dims d, const int flags,
                    float *__restrict__ grad_value, float *__restrict__ grad_loc_arg,
                    float *__restrict__ grad_attw_arg, const int gate, const DetRecords det) {
    using Cfg = BwdCfg<LP, WARPS, TILE_W, QPW>;
    // the raw tensors are passed as float pointers whatever their type, so that the fp32 kernels keep their names
    using PT = ProducerT<V, FUSED>;
    const PT *__restrict__ loc = reinterpret_cast<const PT *>(loc_arg);
    const PT *__restrict__ attw = reinterpret_cast<const PT *>(attw_arg);
    PT *__restrict__ grad_loc = reinterpret_cast<PT *>(grad_loc_arg);
    PT *__restrict__ grad_attw = reinterpret_cast<PT *>(grad_attw_arg);
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ LevelTable lt;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int corner = lane >> 3, chunk = lane & 7;
    uint2 *rec = reinterpret_cast<uint2 *>(smem_raw) + (size_t)warp * 4 * Cfg::kPlane;
    float4 *aux = reinterpret_cast<float4 *>(smem_raw + Cfg::kRecBytes) + (size_t)warp * Cfg::kRecPerWarp;

    fill_level_table(lt, shapes, lstart, d.L, d.P, d.S, d.Lq, Cfg::kGroup, Cfg::kTileH, TILE_W,
                     flags & 1);
    // what-if knob for profiles/ only (WRONG grad_value): drop the reductions of the first
    // `drop_pairs` record pairs of every query, i.e. of the coarsest levels -- the best case any
    // scheme that merges those contributions before they reach L2 could hope for
    const int drop_pairs = flags >> 1;
    __syncthreads();
    // launched next to the merging kernel (msda_bwd_sorted.cu): the shared probe of the locations decides
    if (gate == GATE_RUN_IF_SPREAD && probe_points_stay_local<FUSED>(lt, loc, d.N, d.Lq, d.M, d.L, d.P)) return;

    const int M = d.M;
    const long long items = (long long)d.N * M * lt.groups;
    const uint32_t pix_stride = (uint32_t)M * 8u;

    // which of the L*P points this lane finalises after the first reduce-scatter
    // (lane bits 2,1,0 = chunk bits): index unwinding, see rs_step()
    const bool b2 = chunk & 4, b1 = chunk & 2, b0 = chunk & 1;
    const bool c1 = corner & 2, c0 = corner & 1;

    for (long long item = blockIdx.x; item < items; item += gridDim.x) {
        const int m = (int)(item % M);
        const long long rest = item / M;
        const int g = (int)(rest % lt.groups);
        const long long n = rest / lt.groups;
        int q0, cnt;
        warp_queries(lt, d.L, g, warp, Cfg::kGroup, Cfg::kTileH, TILE_W, d.Lq, Cfg::kQPW, q0, cnt);

        // ---- phase 1: records (one plane per corner) + per-point coefficients ----
        phase1_records<FUSED, LP, Cfg::kQPW, Cfg::kPlane, true>(lt, rec, aux, loc, attw, pr, n, q0, cnt, m, M,
                                                                d.Lq, d.L, pix_stride, (uint32_t)d.S * pix_stride, lane);
        __syncwarp();

        // ---- phase 2 ----
        const long long img = n * (long long)d.S * M * 8 + chunk;
        const V *vb = value + img * 4;
        float4 *gvb = reinterpret_cast<float4 *>(grad_value) + img;
        const uint4 *plane = reinterpret_cast<const uint4 *>(rec + corner * Cfg::kPlane);
        for (int qi = 0; qi < cnt; ++qi) {
            const long long qrow = (n * d.Lq + q0 + qi) * M + m;
            const float4 go = ldg_stream_v4(grad_out + (qrow * 8 + chunk) * 4);
            const uint4 *rq = plane + qi * Cfg::kPairs;
            // RECORDS: this query-head's first slot, and the first grad_value row of image n
            const uint32_t slot0 = (uint32_t)qrow * (uint32_t)(LP * 4) + (uint32_t)corner;
            const uint32_t key0 = (uint32_t)n * (uint32_t)d.S * (uint32_t)M;
            float dpart[LP];
#pragma unroll
            for (int pb = 0; pb < Cfg::kPairs; pb += BATCH) {
                constexpr int kB = BATCH;
                uint4 e[kB];
                float4 va[kB], vc[kB];
#pragma unroll
                for (int j = 0; j < kB; ++j)
                    if (pb + j < Cfg::kPairs) e[j] = lds_u4(rq + pb + j);
#pragma unroll
                for (int j = 0; j < kB; ++j) {                  // 2*BATCH independent loads in flight
                    if (pb + j < Cfg::kPairs) {
                        va[j] = ldg_keep_v4_if(vb, e[j].x);
                        vc[j] = ldg_keep_v4_if(vb, e[j].z);
                    }
                }
#pragma unroll
                for (int j = 0; j < kB; ++j) {
                    if (pb + j < Cfg::kPairs) {
                        const int sp = 2 * (pb + j);
                        const float wa = __uint_as_float(e[j].y), wc = __uint_as_float(e[j].w);
                        if (RECORDS) {
                            if (chunk == 0) {
                                const uint32_t sa = slot0 + (uint32_t)sp * 4u, sc = sa + 4u;
                                // record offsets are (pixel*M + m)*8 float4 from the image start
                                det.key[sa] = e[j].x != kNoCorner ? key0 + (e[j].x >> 3) : det.sentinel;
                                det.key[sc] = e[j].z != kNoCorner ? key0 + (e[j].z >> 3) : det.sentinel;
                                det.slot_id[sa] = sa;
                                det.slot_id[sc] = sc;
                                static_cast<float *>(det.w)[sa] = wa;
                                static_cast<float *>(det.w)[sc] = wc;
                            }
                        } else if (pb + j >= drop_pairs) {
                            red_add_f4_if(gvb, e[j].x, make_float4(wa * go.x, wa * go.y, wa * go.z, wa * go.w));
                            red_add_f4_if(gvb, e[j].z, make_float4(wc * go.x, wc * go.y, wc * go.z, wc * go.w));
                        }
                        const float da = fmaf(va[j].w, go.w, fmaf(va[j].z, go.z, fmaf(va[j].y, go.y, va[j].x * go.x)));
                        const float dc = fmaf(vc[j].w, go.w, fmaf(vc[j].z, go.z, fmaf(vc[j].y, go.y, vc[j].x * go.x)));
                        dpart[sp] = (e[j].x != kNoCorner) ? da : 0.f;      // a corner outside contributes 0
                        dpart[sp + 1] = (e[j].z != kNoCorner) ? dc : 0.f;
                    }
                }
            }
            // D_k for this lane's corner: sum over the 8 chunk lanes (lane bits 2,1,0)
            float r1[Cfg::kN1], r2[Cfg::kN2], r3[Cfg::kN3];
            rs_step<LP>(dpart, r1, b2, 4);
            rs_step<Cfg::kN1>(r1, r2, b1, 2);
            rs_step<Cfg::kN2>(r2, r3, b0, 1);
            // coefficient of D_corner in (d/dx, d/dy, d/dweight) of each finalised point
            float t0[Cfg::kT0];
#pragma unroll
            for (int j = 0; j < Cfg::kN3; ++j) {
                const int i2 = j + (b0 ? Cfg::kN3 : 0);          // index before step 3
                const int i1 = i2 + (b1 ? Cfg::kN2 : 0);         // index before step 2
                const int sp = i1 + (b2 ? Cfg::kN1 : 0);         // index before step 1 = point
                const bool live = (i2 < Cfg::kN2) && (i1 < Cfg::kN1) && (sp < LP);
                float cx = 0.f, cy = 0.f, ca = 0.f;
                if (live) {
                    const float4 a = aux[qi * LP + sp];          // {lh, lw, attention weight, level}
                    const int4 lv = lt.hws[__float_as_int(a.w)];
                    const float lh = a.x, lw = a.y, hh = 1.f - a.x, hw = 1.f - a.y;
                    const float fh = c1 ? lh : hh;               // factor along h of this corner's weight
                    const float fw = c0 ? lw : hw;               // factor along w
                    ca = fh * fw;                                // d val / d weight part (cuh:161)
                    cx = (c0 ? fh : -fh) * (a.z * (float)lv.y);  // W * aw * d w_k / d w  (cuh:128-156,162)
                    cy = (c1 ? fw : -fw) * (a.z * (float)lv.x);  // H * aw * d w_k / d h  (cuh:128-156,163)
                }
                t0[3 * j + 0] = cx * r3[j];
                t0[3 * j + 1] = cy * r3[j];
                t0[3 * j + 2] = ca * r3[j];
            }
            // sum over the 4 corner groups (lane bits 4,3)
            float t1[Cfg::kT1], t2[Cfg::kT2];
            rs_step<Cfg::kT0>(t0, t1, c1, 16);
            rs_step<Cfg::kT1>(t1, t2, c0, 8);
            if constexpr (!FUSED) {
#pragma unroll
                for (int i = 0; i < Cfg::kT2; ++i) {
                    const int u1 = i + (c0 ? Cfg::kT2 : 0);
                    const int u0 = u1 + (c1 ? Cfg::kT1 : 0);
                    if (u1 < Cfg::kT1 && u0 < Cfg::kT0) {
                        const int j = u0 / 3, comp = u0 - 3 * j;
                        const int i2 = j + (b0 ? Cfg::kN3 : 0);
                        const int i1 = i2 + (b1 ? Cfg::kN2 : 0);
                        const int sp = i1 + (b2 ? Cfg::kN1 : 0);
                        if (i2 < Cfg::kN2 && i1 < Cfg::kN1 && sp < LP) {
                            const long long sidx = qrow * LP + sp;
                            if (comp == 2) stg_stream_f1(grad_attw + sidx, t2[i]);
                            else stg_stream_f1(grad_loc + 2 * sidx + comp, t2[i]);
                        }
                    }
                }
            } else {
                // the producers' backward.  Their per-point data is re-read from `aux` here, after the
                // reduce-scatters, instead of being carried through them in registers.
                //   locations: d loc / d offset = 1 / (W, H)  (mod.py:110-112)
                //   softmax:   grad_logit_i = a_i * (ga_i - sum_j a_j * ga_j)  (torch's softmax backward:
                //              (grad - sum(grad * out)) * out); the ga_j sit on different lanes
                int sp_of[Cfg::kT2], comp_of[Cfg::kT2];          // which (point, component) t2[i] is
                float prob[Cfg::kT2], div[Cfg::kT2];
                float dot_a = 0.f;
#pragma unroll
                for (int i = 0; i < Cfg::kT2; ++i) {
                    const int u1 = i + (c0 ? Cfg::kT2 : 0);
                    const int u0 = u1 + (c1 ? Cfg::kT1 : 0);
                    const int j = u0 / 3;
                    const int i2 = j + (b0 ? Cfg::kN3 : 0);
                    const int i1 = i2 + (b1 ? Cfg::kN2 : 0);
                    const int sp = i1 + (b2 ? Cfg::kN1 : 0);
                    const bool live = u1 < Cfg::kT1 && u0 < Cfg::kT0 && i2 < Cfg::kN2 && i1 < Cfg::kN1 && sp < LP;
                    sp_of[i] = live ? sp : -1;
                    comp_of[i] = u0 - 3 * j;
                    prob[i] = 0.f;
                    div[i] = 1.f;
                    if (live) {
                        const float4 a = aux[qi * LP + sp];
                        const int4 lv = lt.hws[__float_as_int(a.w)];
                        prob[i] = a.z;
                        div[i] = (float)(comp_of[i] == 0 ? lv.y : lv.x);
                        if (comp_of[i] == 2) dot_a = fmaf(a.z, t2[i], dot_a);
                    }
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) dot_a += __shfl_xor_sync(kFullMask, dot_a, o);
#pragma unroll
                for (int i = 0; i < Cfg::kT2; ++i) {
                    if (sp_of[i] >= 0) {
                        const long long sidx = qrow * LP + sp_of[i];
                        if (comp_of[i] == 2) stg_stream_v1<PT>(grad_attw + sidx, prob[i] * (t2[i] - dot_a));
                        else stg_stream_v1<PT>(grad_loc + 2 * sidx + comp_of[i], __fdiv_rn(t2[i], div[i]));
                    }
                }
            }
        }
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------
// host side: launch_bwd_d32() serves the plain op, the fused producers (Producers::ref set) and
// the deterministic records (msda_det.cu), the last two in the default CTA shape only
// ---------------------------------------------------------------------------
template <typename V, int LP, int WARPS, int TILE_W, int MIN_CTAS, int BATCH, int QPW, bool FUSED, bool RECORDS>
static cudaError_t launch_bwd_cfg(const V *grad_out, const V *value, const int64_t *shapes, const int64_t *lstart,
                                  const ProducerT<V, FUSED> *loc, const ProducerT<V, FUSED> *attw, const Producers &pr,
                                  const Dims &d, float *grad_value, ProducerT<V, FUSED> *grad_loc,
                                  ProducerT<V, FUSED> *grad_attw, const DetRecords &det, int gate,
                                  cudaStream_t stream) {
    using Cfg = BwdCfg<LP, WARPS, TILE_W, QPW>;
    constexpr auto kern = msda_bwd_d32_kernel<V, LP, WARPS, TILE_W, MIN_CTAS, BATCH, QPW, FUSED, RECORDS>;
    cudaError_t e;
    const int blocks = persistent_blocks<kern>(WARPS * 32, Cfg::kSmem, d, &e);
    if (blocks == 0) return e;
    const int flags = (option_value(OPT_TILE_ORDER) != 1 ? 1 : 0) | (whatif_value(OPT_WHATIF_DROP_REDS) << 1);
    kern<<<blocks, WARPS * 32, Cfg::kSmem, stream>>>(grad_out, value, shapes, lstart, reinterpret_cast<const float *>(loc),
                                                     reinterpret_cast<const float *>(attw), pr, d, flags, grad_value,
                                                     reinterpret_cast<float *>(grad_loc),
                                                     reinterpret_cast<float *>(grad_attw), gate, det);
    note_launch();
    return cudaGetLastError();
}

template <typename V, typename P, int LP>
static cudaError_t launch_bwd_lp(const V *grad_out, const V *value, const int64_t *shapes,
                                 const int64_t *lstart, const P *loc, const P *attw, const Producers &pr,
                                 const Dims &d, float *gv, P *gl, P *gw, const DetRecords *det, int gate,
                                 cudaStream_t st) {
    // variant = (warps, query tile width, min CTAs per SM -> register budget, load batch in pairs,
    //            queries per warp)
#define MSDA_BWD(W, TW, C, B, Q, F, R) \
    launch_bwd_cfg<V, LP, W, TW, C, B, Q, F, R>(grad_out, value, shapes, lstart, loc, attw, pr, d, gv, gl, gw, \
                                             R ? *det : DetRecords{}, gate, st)
    // 16-bit, fused producers and the deterministic records: the default shape only (16-bit fused at L*P = 16: below)
    if constexpr (is16<P>) {          // 16-bit fused producers
        if constexpr (LP == 16)       // 12 warps (85 registers): in the default shape they spill
            return det != nullptr ? MSDA_BWD(12, 16, 2, 1, 8, true, true) : MSDA_BWD(12, 16, 2, 1, 8, true, false);
        else
            return det != nullptr ? MSDA_BWD(16, 16, 2, 1, 8, true, true) : MSDA_BWD(16, 16, 2, 1, 8, true, false);
    } else if constexpr (is16<V>) {   // 16-bit plain
        return det != nullptr ? MSDA_BWD(16, 16, 2, 1, 8, false, true) : MSDA_BWD(16, 16, 2, 1, 8, false, false);
    } else {
    if (det != nullptr)
        return pr.ref != nullptr ? MSDA_BWD(16, 16, 2, 1, 8, true, true) : MSDA_BWD(16, 16, 2, 1, 8, false, true);
    if (pr.ref != nullptr) return MSDA_BWD(16, 16, 2, 1, 8, true, false);
    switch (option_value(OPT_BWD_VARIANT)) {
        case 1: return MSDA_BWD(8, 8, 4, 1, 8, false, false);     //  8 warps, tile  8x8
        case 3: return MSDA_BWD(32, 16, 1, 1, 8, false, false);   // 32 warps, tile 16x16, one CTA per SM
        case 4: return MSDA_BWD(16, 16, 2, 2, 8, false, false);   // 16 warps, 4 loads in flight (spills at 64 regs)
        case 5: return MSDA_BWD(16, 16, 2, 1, 4, false, false);   // 16 warps, tile  4x16, 4 queries per warp (76 KB smem per SM)
        case 6: return MSDA_BWD(8, 8, 2, 6, 8, false, false);     //  8 warps, 114 regs, 12 loads in flight
        case 7: return MSDA_BWD(16, 8, 2, 1, 4, false, false);    // 16 warps, tile  8x8,  4 queries per warp
        case 8: return MSDA_BWD(32, 16, 1, 1, 4, false, false);   // 32 warps, tile  8x16, 4 queries per warp, one CTA per SM
        case 2:
        default: return MSDA_BWD(16, 16, 2, 1, 8, false, false);  // 16 warps, tile  8x16, 8 queries per warp (147 KB smem per SM)
    }
    }
#undef MSDA_BWD
}

// pr.ref == nullptr: plain; otherwise fused producers, gradients w.r.t. the raw sampling offsets (`loc`) and
// attention logits (`attw`).  P: element type of `loc` / `attw` / `gl` / `gw` -- float, or V for the 16-bit fused
// producers.  det != nullptr: deterministic mode (msda_det.cu), grad_value `gv` is not touched and
// the corner records go to `det`.  `gate`: see msda_bwd_sorted.cu.  `handled` = false: the problem is outside
// d32_applies() and nothing was launched.
template <typename V, typename P>
cudaError_t launch_bwd_d32(const V *grad_out, const V *value, const int64_t *shapes, const int64_t *lstart,
                           const P *loc, const P *attw, const Producers &pr, const Dims &d, float *gv,
                           P *gl, P *gw, const DetRecords *det, int gate, cudaStream_t st, bool *handled) {
    *handled = d32_applies(d);
    if (!*handled) return cudaSuccess;
    switch (d.L * d.P) {       // 4, 8, 12 or 16 (d32_applies)
        case 4: return launch_bwd_lp<V, P, 4>(grad_out, value, shapes, lstart, loc, attw, pr, d, gv, gl, gw, det, gate, st);
        case 8: return launch_bwd_lp<V, P, 8>(grad_out, value, shapes, lstart, loc, attw, pr, d, gv, gl, gw, det, gate, st);
        case 12: return launch_bwd_lp<V, P, 12>(grad_out, value, shapes, lstart, loc, attw, pr, d, gv, gl, gw, det, gate, st);
        default: return launch_bwd_lp<V, P, 16>(grad_out, value, shapes, lstart, loc, attw, pr, d, gv, gl, gw, det, gate, st);
    }
}

#define MSDA_BWD_D32(V, P)                                                                                       \
    template cudaError_t launch_bwd_d32<V, P>(const V *, const V *, const int64_t *, const int64_t *, const P *, \
                                              const P *, const Producers &, const Dims &, float *, P *, P *,     \
                                              const DetRecords *, int, cudaStream_t, bool *);
MSDA_BWD_D32(float, float)
MSDA_BWD_D32(__nv_bfloat16, float)
MSDA_BWD_D32(__half, float)
MSDA_BWD_D32(__nv_bfloat16, __nv_bfloat16)
MSDA_BWD_D32(__half, __half)
#undef MSDA_BWD_D32

}  // namespace msda
