// msda_bwd_sorted.cu -- backward MSDA kernel for sm_100a (32 channels per head; fp32 value rows, or bf16 / fp16
// ones with fp32 sums and an fp32 grad_value accumulation buffer) that merges
// the grad_value contributions of a query tile INSIDE the SM before anything is sent to L2.
//
// Replaces ms_deformable_col2im_gpu_kernel_shm_blocksize_aware_reduce_v1<T,32>
// (ms_deform_im2col_cuda.cuh:306-408) and ms_deform_attn_col2im_bilinear (cuh:92-164), where
// every one of the 48 corner rows of a (query, head) goes to L2 as 32 scalar atomicAdds
// (cuh:130-157).  msda_bwd.cu already turned those into one 128-bit reduction per lane, but
// every corner row still travelled to L2 alone: 3.86 GB of reductions per launch for 88 MB of
// grad_value at BASELINE configs[1], pinned at the 6.4 TB/s the L2 reduction path sustains
// (profiles/r1_microbench.txt).  Neighbouring queries of the encoder sample the same pixels
// (their reference points are their own pixel centres, msdeformattn.py:152-166), so here the
// corner records of a tile of 128 queries are SORTED BY DESTINATION PIXEL in shared memory and
// every run of equal pixels is accumulated in registers and sent to L2 once.
//
// One work item = (image n, head m, tile of 128 queries = 8 x 16 pixels of one level).  Per item:
//   pass A   one sampling point per thread: decompose() (the same single home of the integer
//            work as every other kernel), and for each contributing corner whose pixel lies in
//            the item's per-level WINDOW (tile footprint +- 7 px, clipped to the level) the
//            counter of that pixel is incremented (integer shared-memory atomics: 0.84 cycles
//            per warp instruction measured; fp32 ones are CAS loops).  The point's window slots,
//            first pixel, fractions and weight stay in registers for pass B;
//   scan     exclusive prefix sum of the counters (conflict-free warp scans);
//   pass B   every corner record {pixel:18 | query:7 | - | point*4+corner:6, bilinear*attention
//            weight} is written to its sorted position (atomicAdd on the counter returns the
//            rank); corners outside every window are appended behind the sorted ones -- they
//            are processed by the same loop as runs of length one, so correctness never
//            depends on the windows, only the amount of merging does;
//   merge    the record array is cut into equal slices, one per GW-lane group (GW = 4 shipped: a lane owns
//            two 16-byte chunks of a 128-byte row; GW = 8: one), slices interleaved over the warps.  A
//            group walks its slice: at the first record of a pixel it loads that pixel's value row ONCE,
//            then per record reads the query's grad_output row from shared memory, accumulates
//            weight * grad_output in registers (packed fma.rn.f32x2) and forms its part of the dot
//            product D = <value row, grad_output row>; when the pixel changes the accumulator leaves as
//            ONE red.global.add.v4.f32 per lane and chunk.  A run cut by a slice boundary is simply
//            flushed by both groups.  The partial dot products of a body of records are summed over the
//            group's lanes with a shuffle reduce-scatter and land in D[query][point][corner] in shared
//            memory;
//   epilogue one sampling point per thread again: grad_attn_weight and grad_sampling_loc are the
//            reference's linear combinations of the point's four D (cuh:128-163), written with
//            coalesced stores.  Both are deterministic and need no zero fill.
//
// Per (query, head) the L1/shared-memory data pipe now carries 48 grad_output rows + the value
// rows and reductions of the DISTINCT pixels (48 / merge factor, ~9x at configs[1]) instead of
// 48 value rows + 48 reductions; see DESIGN.md section 4.3 for the measured numbers.
//
// Used when the queries are the value pixels (Lq == S, encoder self-attention); when the level
// layout does not tile them (decided on the device, like the other kernels) the windows are
// empty and every record takes the run-of-one path.  Other shapes: msda_bwd.cu.
#include "msda_common.cuh"

namespace msda {

constexpr int kSortTileMax = 256;        // queries per item: 7 or 8 bits of the record word
constexpr int kSortMargin = 7;           // window = tile footprint +- this many pixels (5..7 measured equal, 9: +0.8 %, 4: +2 %)
constexpr uint32_t kNoKey = 0x3ffffu;    // pixel field of an absent record (7-bit query slot); S < kNoKey (host check)
constexpr uint32_t kSlotNone = 0xffffu;  // pass A -> pass B: corner does not contribute
constexpr uint32_t kSlotTail = 0xfffeu;  //                   corner outside every window

// record word: [pixel:18 | query slot:7 | 0 | point*4+corner:6] (tiles of up to 128 queries; 256: pixel:17,
// query slot:8); (word & kQMask) = query slot * 128, the byte offset of the query's grad_output row in
// shared memory
__device__ __forceinline__ uint32_t rec_word(uint32_t pix, uint32_t q, uint32_t pc, int pix_shift) {
    return (pix << pix_shift) | (q << 7) | pc;
}

// TILE_Q queries per item (a TILE_W-wide 2-D tile of one level), SLOTS window pixels per item
template <int LP, int WARPS, int TILE_W, int TILE_Q, int SLOTS>
struct SortCfg {
    static constexpr int kSortTile = TILE_Q, kSortSlots = SLOTS;
    static constexpr int kQBits = TILE_Q > 128 ? 8 : 7;
    static constexpr int kPixShift = 7 + kQBits;                          // record word layout
    static constexpr uint32_t kQMask = ((1u << kQBits) - 1u) << 7;
    static constexpr uint32_t kNoPix = 0xffffffffu >> kPixShift;          // pixel field of an absent record
    static constexpr int kThreads = WARPS * 32;
    static constexpr int kTileH = kSortTile / TILE_W;
    static constexpr int kPC = LP * 4;                       // corner records per query
    static constexpr int kRecs = kSortTile * kPC;            // record capacity of an item
    static constexpr int kPoints = kSortTile * LP;
    static constexpr int kRounds = (kPoints + kThreads - 1) / kThreads;
    static constexpr size_t kRecBytes = (size_t)kRecs * sizeof(uint2);
    static constexpr size_t kGoBytes = (size_t)kSortTile * 128;
    static constexpr size_t kDBytes = (size_t)kRecs * sizeof(float);
    static constexpr size_t kCntBytes = (size_t)kSortSlots * sizeof(uint32_t);
    static constexpr size_t kSmem = kRecBytes + kGoBytes + kDBytes + kCntBytes;
    static_assert(kPC <= 64 && kSortTile % TILE_W == 0, "record word: 6 bits of point*4+corner");
    static_assert(kSortSlots < (int)kSlotTail, "16-bit slot numbers between the passes");
    static_assert(TILE_Q <= kSortTileMax, "8-bit query slot");
};

// where the queries of a tile live
struct TileMap {
    int spatial;        // 1: 2-D tile of level lq; 0: 128 consecutive queries
    int X0, Y0;         // pixel origin of the tile inside its level (spatial)
    int H, W, start;    // of the tile's level
    int q0;             // first query (non-spatial)
};

template <int TILE_W, int TILE_H>
__device__ __forceinline__ TileMap tile_of(const LevelTable &lt, int L, int g) {
    TileMap t;
    t.spatial = lt.spatial;
    t.X0 = 0; t.Y0 = 0; t.H = 0; t.W = 0; t.start = 0;
    t.q0 = g * (TILE_W * TILE_H);
    if (lt.spatial) {
        int l = 0;
        while (l + 1 < L && g >= lt.tile_begin[l + 1]) ++l;
        const int r = g - lt.tile_begin[l];
        const int ty = r / lt.tiles_x[l], tx = r - ty * lt.tiles_x[l];
        t.X0 = tx * TILE_W;
        t.Y0 = ty * TILE_H;
        t.H = lt.H[l];
        t.W = lt.W[l];
        t.start = lt.start[l];
    }
    return t;
}

// query index (inside one image) of slot q of the tile, -1 when the slot is empty
template <int TILE_W>
__device__ __forceinline__ int tile_query(const TileMap &t, int q, int Lq) {
    if (t.spatial) {
        const int y = t.Y0 + q / TILE_W, x = t.X0 + q % TILE_W;
        return (y < t.H && x < t.W) ? t.start + y * t.W + x : -1;
    }
    const int qg = t.q0 + q;
    return qg < Lq ? qg : -1;
}

// Windows of the item whose tile is `t` (warp 0, lane = level): {x0, y0, width | height << 16,
// first slot}; total slots -> *slots_out.  Heuristic only: a window decides which records can be
// merged, never what is computed.
template <int TILE_W, int TILE_H, int kSortSlots>
__device__ __forceinline__ void compute_windows(const LevelTable &lt, int L, const TileMap &t,
                                                int4 *win_out, int *slots_out, int lane) {
    int x0 = 0, y0 = 0, ww = 0, wh = 0;
    if (t.spatial && lane < L) {
        const int Wl = lt.W[lane], Hl = lt.H[lane];
        const float sx = (float)Wl / (float)t.W, sy = (float)Hl / (float)t.H;
        const int X1 = min(t.X0 + TILE_W, t.W), Y1 = min(t.Y0 + TILE_H, t.H);
        int xa = (int)floorf((float)t.X0 * sx) - kSortMargin, xb = (int)ceilf((float)X1 * sx) + kSortMargin;
        int ya = (int)floorf((float)t.Y0 * sy) - kSortMargin, yb = (int)ceilf((float)Y1 * sy) + kSortMargin;
        xa = max(xa, 0); ya = max(ya, 0);
        xb = min(xb, Wl); yb = min(yb, Hl);
        ww = max(xb - xa, 0); wh = max(yb - ya, 0);
        x0 = xa; y0 = ya;
        if ((long long)ww * wh > kSortSlots) { ww = 0; wh = 0; }   // cannot fit on its own
    }
    int area = ww * wh;
    // budget: drop the largest windows (the least merging per slot) until the rest fits
    for (int round = 0; round < kMaxLevels; ++round) {
        int total = area, mx = area;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            total += __shfl_xor_sync(kFullMask, total, o);
            mx = max(mx, __shfl_xor_sync(kFullMask, mx, o));
        }
        if (total <= kSortSlots) break;
        const unsigned who = __ballot_sync(kFullMask, area == mx);
        if (lane == __ffs(who) - 1) { ww = 0; wh = 0; area = 0; }
    }
    int incl = area;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int up = __shfl_up_sync(kFullMask, incl, o);
        if (lane >= o) incl += up;
    }
    if (lane < L) win_out[lane] = make_int4(x0, y0, ww | (wh << 16), incl - area);
    if (lane == 31) *slots_out = incl;
}

// What pass A leaves in registers for pass B, per sampling point.
struct Binned {
    uint32_t s01, s23;     // window slot of each corner (16 bits each), kSlotNone / kSlotTail
    int pix0;              // pixel of corner 0 (row above / column left of the sample)
    float lh, lw, aw;
};

// Pass A for one point: geometry, window slots, per-pixel counts.
// `cnt_s`: the counters' 32-bit shared address (kept in a register by the caller: generic pointers
// make ptxas rebuild the shared-window base at every access)
__device__ __forceinline__ Binned count_point(const LevelTable &lt, const int4 *win, uint32_t cnt_s,
                                              float x, float y, float aw, int p, int kSortSlots) {
    Binned b;
    b.s01 = b.s23 = kSlotNone | (kSlotNone << 16);
    b.pix0 = 0; b.lh = 0.f; b.lw = 0.f; b.aw = aw;
    const int l = lt.level_of[p];
    const int4 lv = lt.hws[l];                       // {H, W, start, -}
    const Geom<float> gm = decompose(x, y, lv.x, lv.y);
    if (gm.cmask == 0) return b;                     // point outside (cuh:293): no record
    const int4 wn = win[l];
    const int ww = wn.z & 0xffff, wh = wn.z >> 16;
    const int sx = gm.w_low - wn.x, sy = gm.h_low - wn.y;
    b.pix0 = lv.z + gm.h_low * lv.y + gm.w_low;      // h_low / w_low may be -1: only used with a valid corner
    b.lh = gm.lh; b.lw = gm.lw;
    uint32_t sl[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int dx = k & 1, dy = k >> 1;
        sl[k] = kSlotNone;
        if (gm.cmask & (1 << k)) {
            const bool inwin = (unsigned)(sx + dx) < (unsigned)ww && (unsigned)(sy + dy) < (unsigned)wh;
            sl[k] = kSlotTail;
            if (inwin) {
                const int slot = wn.w + (sy + dy) * ww + sx + dx;
#ifdef MSDA_CHECK_BOUNDS
                assert(slot >= 0 && slot < kSortSlots);
#else
                (void)kSortSlots;
#endif
                asm volatile("red.shared.add.u32 [%0], 1;" ::"r"(cnt_s + 4u * (uint32_t)slot) : "memory");
                sl[k] = (uint32_t)slot;
            }
        }
    }
    b.s01 = sl[0] | (sl[1] << 16);
    b.s23 = sl[2] | (sl[3] << 16);
    return b;
}

// Pass B for one point: its corner records to their places.  `wbase` = query slot << 7 | point * 4.
__device__ __forceinline__ void place_point(const Binned &b, uint32_t cnt_s, uint32_t rec_s, uint32_t *tail_ctr,
                                            uint32_t n_in, int W, uint32_t wbase, int S, int rec_cap, int pix_shift) {
    const float hh = 1.f - b.lh, hw = 1.f - b.lw;
    const float wk[4] = {(hh * hw) * b.aw, (hh * b.lw) * b.aw, (b.lh * hw) * b.aw, (b.lh * b.lw) * b.aw};   // bilinear * attention
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int dx = k & 1, dy = k >> 1;
        const uint32_t pair = dy ? b.s23 : b.s01;
        const uint32_t slot = dx ? (pair >> 16) : (pair & 0xffffu);
        if (slot != kSlotNone) {
            uint32_t pos;
            if (slot != kSlotTail)
                asm volatile("atom.shared.add.u32 %0, [%1], 1;" : "=r"(pos) : "r"(cnt_s + 4u * slot) : "memory");
            else
                pos = n_in + atomicAdd(tail_ctr, 1u);
            const int pix = b.pix0 + dy * W + dx;
#ifdef MSDA_CHECK_BOUNDS
            assert(pix >= 0 && pix < S && (int)pos < rec_cap);
#else
            (void)S; (void)rec_cap;
#endif
            asm volatile("st.shared.v2.u32 [%0], {%1,%2};" ::"r"(rec_s + 8u * pos),
                         "r"(((uint32_t)pix << pix_shift) | wbase | (uint32_t)k), "r"(__float_as_uint(wk[k])) : "memory");
        }
    }
}

// shared-memory accesses by 32-bit shared address (no generic-address arithmetic in the merge loop)
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint2 lds_u2(uint32_t a) {
    uint2 r;
    asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "r"(a) : "memory");
    return r;
}
__device__ __forceinline__ uint32_t lds_u1(uint32_t a) {
    uint32_t r;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(r) : "r"(a) : "memory");
    return r;
}
__device__ __forceinline__ float4 lds_f4(uint32_t a) {
    float4 r;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "r"(a) : "memory");
    return r;
}
// packed fp32x2 arithmetic (SASS FFMA2 / FMUL2): two IEEE fp32 operations per instruction on a
// 64-bit register pair {lo, hi}
__device__ __forceinline__ void ffma2_bcast(uint64_t &acc, uint32_t w_bits, uint64_t g) {   // acc += {w, w} * g
    asm("{\n\t.reg .b64 rw;\n\tmov.b64 rw, {%1,%1};\n\tfma.rn.f32x2 %0, rw, %2, %0;\n\t}" : "+l"(acc) : "r"(w_bits), "l"(g));
}
// {x, y} = {w, w} * g
__device__ __forceinline__ void fmul2_bcast_xy(float &x, float &y, uint32_t w_bits, uint64_t g) {
    asm("{\n\t.reg .b64 rw, ra;\n\tmov.b64 rw, {%2,%2};\n\tmul.rn.f32x2 ra, rw, %3;\n\tmov.b64 {%0,%1}, ra;\n\t}"
        : "=f"(x), "=f"(y) : "r"(w_bits), "l"(g));
}
// {x, y} += {w, w} * g on two adjacent floats of a float4 accumulator (an aligned register pair)
__device__ __forceinline__ void ffma2_bcast_xy(float &x, float &y, uint32_t w_bits, uint64_t g) {
    asm("{\n\t.reg .b64 rw, ra;\n\tmov.b64 rw, {%2,%2};\n\tmov.b64 ra, {%0,%1};\n\t"
        "fma.rn.f32x2 ra, rw, %3, ra;\n\tmov.b64 {%0,%1}, ra;\n\t}" : "+f"(x), "+f"(y) : "r"(w_bits), "l"(g));
}
__device__ __forceinline__ void ffma2_p(uint64_t &acc, uint64_t a, uint64_t b) {            // acc += a * b
    asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc) : "l"(a), "l"(b));
}
__device__ __forceinline__ uint64_t fmul2_p(uint64_t a, uint64_t b) {
    uint64_t d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ uint64_t fadd2_p(uint64_t a, uint64_t b) {
    uint64_t d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ float sum2(uint64_t a) {
    float lo, hi;
    asm("mov.b64 {%0,%1}, %2;" : "=f"(lo), "=f"(hi) : "l"(a));
    return lo + hi;
}
__device__ __forceinline__ void lds_2x64(uint32_t a, uint64_t &x, uint64_t &y) {
    asm volatile("ld.shared.v2.b64 {%0,%1}, [%2];" : "=l"(x), "=l"(y) : "r"(a) : "memory");
}
__device__ __forceinline__ void ldg_2x64(const char *p, uint64_t &x, uint64_t &y) {
    asm volatile("ld.global.nc.v2.b64 {%0,%1}, [%2];" : "=l"(x), "=l"(y) : "l"(p));
}
__device__ __forceinline__ void red_2x64(char *p, uint64_t x, uint64_t y) {
    asm volatile("{\n\t.reg .f32 a, b, c, d;\n\tmov.b64 {a,b}, %1;\n\tmov.b64 {c,d}, %2;\n\t"
                 "red.global.add.v4.f32 [%0], {a,b,c,d};\n\t}" ::"l"(p), "l"(x), "l"(y) : "memory");
}
template <typename P>
__device__ __forceinline__ P xor64(P p) {       // the other 64-byte half of a 128-byte aligned row
    return reinterpret_cast<P>(reinterpret_cast<uintptr_t>(p) ^ (uintptr_t)64);
}
// a lane's 4-channel chunk of a value row as two packed fp32 pairs (16-bit V: 8 bytes, widened)
template <typename V>
__device__ __forceinline__ void ldg_value_chunk(const char *p, uint64_t &x, uint64_t &y) {
    if constexpr (!is16<V>) {
        ldg_2x64(p, x, y);
    } else {
        uint2 u;
        asm volatile("ld.global.nc.v2.u32 {%0,%1}, [%2];" : "=r"(u.x), "=r"(u.y) : "l"(p));
        const float4 f = widen4<V>(u);
        x = (uint64_t)__float_as_uint(f.x) | ((uint64_t)__float_as_uint(f.y) << 32);
        y = (uint64_t)__float_as_uint(f.z) | ((uint64_t)__float_as_uint(f.w) << 32);
    }
}
template <typename V>
__device__ __forceinline__ const char *other_half(const char *p) {   // the chunk 4 chunks away in an aligned row
    return reinterpret_cast<const char *>(reinterpret_cast<uintptr_t>(p) ^ (uintptr_t)(4 * kChunkBytes<V>));
}
__device__ __forceinline__ void sts_f1(uint32_t a, float v) {
    asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory");
}
__device__ __forceinline__ void red_add_f4(float4 *p, const float4 v) {
    asm volatile("red.global.add.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// GW: lanes per record in the merge loop (8: 16 bytes of a row per lane, 4: 32 bytes)
// FUSED: `loc` / `attw` are the raw sampling offsets / attention logits and `grad_loc` / `grad_attw`
//      receive the gradients with respect to THEM (SURVEY 8f.1, as in msda_bwd.cu): pass A forms
//      location = ref + offset / (W, H) and the softmax of the (query, head)'s L*P logits (exchanged
//      through shared memory), the epilogue applies 1 / (W, H) and the softmax backward.
// V: element type of grad_out / value.  16-bit: the grad_output tile is widened to fp32 while it is staged (the merge
// loop reads it as for fp32), a lane's value chunk is 8 bytes of a 64-byte row, and grad_value is the fp32
// accumulation buffer (128-byte rows, as for fp32).  FUSED with 16-bit V: the raw offsets / logits and their
// gradients are of type V too (ProducerT), widened in pass A and the epilogue, rounded once as they are stored
template <typename V, int LP, int WARPS, int TILE_W, int MIN_CTAS, int TILE_Q, int SLOTS, int GW, bool FUSED>
__global__ void __launch_bounds__(WARPS * 32, MIN_CTAS)
msda_bwd_sorted_kernel(const V *__restrict__ grad_out, const V *__restrict__ value,
                       const int64_t *__restrict__ shapes, const int64_t *__restrict__ lstart,
                       const float *__restrict__ loc_arg, const float *__restrict__ attw_arg, const Producers pr,
                       const Dims d, const int flags, float *__restrict__ grad_value,
                       float *__restrict__ grad_loc_arg, float *__restrict__ grad_attw_arg, const int gate) {
    using Cfg = SortCfg<LP, WARPS, TILE_W, TILE_Q, SLOTS>;
    // the raw tensors are passed as float pointers whatever their type, so that the fp32 kernels keep their names
    using PT = ProducerT<V, FUSED>;
    const PT *__restrict__ loc = reinterpret_cast<const PT *>(loc_arg);
    const PT *__restrict__ attw = reinterpret_cast<const PT *>(attw_arg);
    PT *__restrict__ grad_loc = reinterpret_cast<PT *>(grad_loc_arg);
    PT *__restrict__ grad_attw = reinterpret_cast<PT *>(grad_attw_arg);
    constexpr int NT = Cfg::kThreads;
    constexpr int kSortTile = Cfg::kSortTile, kSortSlots = Cfg::kSortSlots;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ LevelTable lt;
    __shared__ int4 win[2][kMaxLevels];
    __shared__ int win_slots[2];
    __shared__ uint32_t warp_tot[WARPS];
    __shared__ uint32_t tail_ctr;

    uint2 *rec = reinterpret_cast<uint2 *>(smem_raw);
    float4 *go_sm = reinterpret_cast<float4 *>(smem_raw + Cfg::kRecBytes);
    float *dsm = reinterpret_cast<float *>(smem_raw + Cfg::kRecBytes + Cfg::kGoBytes);
    uint32_t *cnt = reinterpret_cast<uint32_t *>(smem_raw + Cfg::kRecBytes + Cfg::kGoBytes + Cfg::kDBytes);
    // FUSED: softmax weight of every point of the item, pass A -> epilogue (entry s is private to the
    // thread that owns point s); logits / weighted gradients are exchanged through the record array,
    // which is free in pass A and after the merge: two disjoint pieces, see the barriers' comments
    float *aw_sm = reinterpret_cast<float *>(smem_raw + Cfg::kSmem);
    float *scr_a = reinterpret_cast<float *>(rec), *scr_e = scr_a + Cfg::kPoints, *scr_x = scr_a + 2 * Cfg::kPoints;
    static_assert(!FUSED || (LP % 4 == 0 && 3 * Cfg::kPoints * sizeof(float) <= Cfg::kRecBytes), "softmax scratch");

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    fill_level_table(lt, shapes, lstart, d.L, d.P, d.S, d.Lq, kSortTile, Cfg::kTileH, TILE_W, flags & 1);
    for (int i = tid; i < kSortSlots; i += NT) cnt[i] = 0u;   // invariant: zero outside pass A .. pass B
    __syncthreads();
    // launched next to the per-row reduction kernel: the shared probe of the locations decides
    if (gate == GATE_RUN_IF_LOCAL && !probe_points_stay_local<FUSED>(lt, loc, d.N, d.Lq, d.M, d.L, d.P)) return;

    const int M = d.M, L = d.L, Lq = d.Lq;
    const long long items = (long long)d.N * M * lt.groups;

    long long item = blockIdx.x;
    if (warp == 0 && item < items) {
        const TileMap t0 = tile_of<TILE_W, Cfg::kTileH>(lt, L, (int)((item / M) % lt.groups));
        compute_windows<TILE_W, Cfg::kTileH, Cfg::kSortSlots>(lt, L, t0, win[0], &win_slots[0], lane);
    }
    __syncthreads();

    for (int buf = 0; item < items; item += gridDim.x, buf ^= 1) {
        const int m = (int)(item % M);
        const long long rest = item / M;
        const int g = (int)(rest % lt.groups);
        const long long n = rest / lt.groups;
        const int4 *wn = win[buf];
        const int nslots = win_slots[buf];
        if (tid == 0) tail_ctr = 0u;
        // rows of image n: 64-bit bases here, 32-bit offsets (query * M + m) * {8, LP} below
        // (Lq * M * 16 < 2^32: host check)
        const V *go_n = grad_out + n * Lq * (long long)M * 32;
        const Pair<PT> *loc_n = reinterpret_cast<const Pair<PT> *>(loc) + n * Lq * (long long)M * LP;
        const PT *attw_n = attw + n * Lq * (long long)M * LP;

        uint32_t n_in;
        {
            const TileMap tm = tile_of<TILE_W, Cfg::kTileH>(lt, L, g);
            uint32_t cnt_s = smem_u32(cnt), rec_sa = smem_u32(rec);
            asm volatile("" : "+r"(cnt_s), "+r"(rec_sa));          // live in registers, not re-derived per access
            // ---- the tile's grad_output rows -> shared memory (read once per record in the merge):
            // asynchronous copies, waited for at the end of pass B; empty query slots are zero-filled ----
            {
                const uint32_t go_dst = smem_u32(go_sm);
                if constexpr (!is16<V>) {
#pragma unroll
                    for (int i = tid; i < kSortTile * 8; i += NT) {
                        const int qg = tile_query<TILE_W>(tm, i >> 3, Lq);
                        const float4 *src = reinterpret_cast<const float4 *>(go_n) +
                                            (qg >= 0 ? (uint32_t)(qg * M + m) * 8u + (uint32_t)(i & 7) : 0u);
                        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;"
                                     ::"r"(go_dst + 16u * (uint32_t)i), "l"(src), "r"(qg >= 0 ? 16 : 0) : "memory");
                    }
                    asm volatile("cp.async.commit_group;" ::: "memory");
                } else {
                    // 16-bit: widened while staging (synchronous: all loads issued before the first store).  Measured
                    // faster than staging the 16-bit rows with cp.async (8 KB) and widening them in the merge loop:
                    // bf16, merging kernel, 0.599 against 0.622 ms at configs[1], 2.44 against 2.58 ms at the
                    // configs[2] shape (DESIGN.md section 11, profiles/r5_staging.jsonl)
                    constexpr int kPer = (kSortTile * 8 + NT - 1) / NT;
                    float4 gs[kPer];
#pragma unroll
                    for (int k = 0; k < kPer; ++k) {
                        const int i = tid + k * NT;
                        const int qg = i < kSortTile * 8 ? tile_query<TILE_W>(tm, i >> 3, Lq) : -1;
                        gs[k] = qg >= 0 ? ldg_stream_v4(at_chunk(go_n, (uint32_t)(qg * M + m) * 8u + (uint32_t)(i & 7)))
                                        : make_float4(0.f, 0.f, 0.f, 0.f);
                    }
#pragma unroll
                    for (int k = 0; k < kPer; ++k) {
                        const int i = tid + k * NT;
                        if (i < kSortTile * 8)
                            asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};"
                                         ::"r"(go_dst + 16u * (uint32_t)i), "f"(gs[k].x), "f"(gs[k].y), "f"(gs[k].z),
                                           "f"(gs[k].w) : "memory");
                    }
                }
            }

            // ---- pass A: load the points, count the in-window corners per pixel ----
            Binned bn[Cfg::kRounds];
            bool live[Cfg::kRounds];
            {
                float px[Cfg::kRounds], py[Cfg::kRounds], pw[Cfg::kRounds];
                float2 rp[FUSED ? Cfg::kRounds : 1];           // FUSED: the query's reference point in the point's level
#pragma unroll
                for (int r = 0; r < Cfg::kRounds; ++r) {       // all global loads first
                    const int s = r * NT + tid;
                    const int q = s / LP, p = s - q * LP;
                    live[r] = false;
                    px[r] = 0.f; py[r] = 0.f; pw[r] = 0.f;
                    if (FUSED) rp[r] = make_float2(0.f, 0.f);
                    if (s < Cfg::kPoints) {
                        const int qg = tile_query<TILE_W>(tm, q, Lq);
                        if (qg >= 0) {
                            const uint32_t row = (uint32_t)(qg * M + m) * (uint32_t)LP + (uint32_t)p;
                            const float2 xy = ldg_stream_pair<PT>(loc_n + row);
                            px[r] = xy.x; py[r] = xy.y;
                            pw[r] = ldg_stream_one<PT>(attw_n + row);
                            if (FUSED)
                                rp[r] = ldg_stream_f2(reinterpret_cast<const float2 *>(
                                    pr.ref + n * pr.ref_bstride + ((long long)qg * L + lt.level_of[p]) * 2));
                            live[r] = true;
                        }
                    }
                }
                if (FUSED) {
                    // softmax over each (query, head)'s LP logits (mod.py:107-108) and the locations
                    // ref + offset / (W, H) (mod.py:110-112), with the arithmetic of phase1_records()
                    // (msda_common.cuh): same max / sum tree, same exact division -> the same bits
#pragma unroll
                    for (int r = 0; r < Cfg::kRounds; ++r)
                        if (live[r]) scr_a[r * NT + tid] = pw[r];
                    __syncthreads();                                        // logits of the item visible
                    float ex[Cfg::kRounds];
#pragma unroll
                    for (int r = 0; r < Cfg::kRounds; ++r) {                // row maximum, own exponential
                        const int s = r * NT + tid;
                        ex[r] = 0.f;
                        if (live[r]) {
                            const float *row = scr_a + (s / LP) * LP;
                            float mx = row[0];
#pragma unroll
                            for (int j = 1; j < LP; ++j) mx = fmaxf(mx, row[j]);
                            ex[r] = expf(pw[r] - mx);
                            scr_x[s] = ex[r];
                        }
                    }
                    __syncthreads();                                        // exponentials of the item visible
#pragma unroll
                    for (int r = 0; r < Cfg::kRounds; ++r) {
                        const int s = r * NT + tid;
                        const int q = s / LP, p = s - q * LP;
                        if (live[r]) {
                            const float *row = scr_x + q * LP;
                            float part[4];                                  // the summation tree of phase1_records()
#pragma unroll
                            for (int k = 0; k < 4; ++k) {
                                part[k] = 0.f;
#pragma unroll
                                for (int j = 0; j < LP / 4; ++j) part[k] += row[k * (LP / 4) + j];
                            }
                            pw[r] = __fdiv_rn(ex[r], (part[0] + part[1]) + (part[2] + part[3]));
                            aw_sm[s] = pw[r];
                            const int l = lt.level_of[p];
                            const float2 rc = lt.rcp_wh[l];
                            px[r] = rp[r].x + div_by_size(px[r], (float)lt.W[l], rc.x);
                            py[r] = rp[r].y + div_by_size(py[r], (float)lt.H[l], rc.y);
                        }
                    }
                }
#pragma unroll
                for (int r = 0; r < Cfg::kRounds; ++r) {
                    const int s = r * NT + tid;
                    const int p = s % LP;
                    bn[r].s01 = bn[r].s23 = kSlotNone | (kSlotNone << 16);
                    if (live[r])
                        bn[r] = count_point(lt, wn, cnt_s, px[r], py[r], pw[r], p, Cfg::kSortSlots);
                }
            }
            __syncthreads();                                                // B1: counts complete

            // ---- exclusive scan of the pixel counters ----
            const int wpw = (((nslots + WARPS - 1) / WARPS) + 31) & ~31;    // counters per warp, multiple of 32
            const int wbeg = warp * wpw, wend = min(wbeg + wpw, nslots);
            {
                uint32_t sum = 0;
                for (int w = wbeg + lane; w < wend; w += 32) sum += cnt[w];
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(kFullMask, sum, o);
                if (lane == 0) warp_tot[warp] = sum;
            }
            __syncthreads();                                                // B2: warp totals
            {
                const uint32_t wt = lane < WARPS ? warp_tot[lane] : 0u;
                uint32_t incl = wt;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const uint32_t up = __shfl_up_sync(kFullMask, incl, o);
                    if (lane >= o) incl += up;
                }
                n_in = __shfl_sync(kFullMask, incl, 31);
                uint32_t run = __shfl_sync(kFullMask, incl - wt, warp);     // records before this warp's counters
                for (int w0 = wbeg; w0 < wend; w0 += 32) {
                    const int w = w0 + lane;
                    const uint32_t c = w < wend ? cnt[w] : 0u;
                    uint32_t inc = c;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {
                        const uint32_t up = __shfl_up_sync(kFullMask, inc, o);
                        if (lane >= o) inc += up;
                    }
                    if (w < wend) cnt[w] = run + inc - c;
                    run += __shfl_sync(kFullMask, inc, 31);
                }
            }
            __syncthreads();                                                // B3: offsets complete

            // ---- pass B: records to their sorted positions (outside every window: appended) ----
#pragma unroll
            for (int r = 0; r < Cfg::kRounds; ++r) {
                const int s = r * NT + tid;
                const int q = s / LP, p = s - q * LP;
                if ((bn[r].s01 & bn[r].s23) != (kSlotNone | (kSlotNone << 16)))
                    place_point(bn[r], cnt_s, rec_sa, &tail_ctr, n_in, lt.W[lt.level_of[p]],
                                ((uint32_t)q << 7) | (uint32_t)(p * 4), d.S, Cfg::kRecs, Cfg::kPixShift);
            }
            if constexpr (!is16<V>) asm volatile("cp.async.wait_group 0;" ::: "memory");
        }
        __syncthreads();                                                    // B4: records + grad_output tile complete

        // counters back to zero for the next item; warp 0 prepares the next item's windows
        for (int i = tid; i < nslots; i += NT) cnt[i] = 0u;
        if (warp == 0 && item + gridDim.x < items) {
            const TileMap tn = tile_of<TILE_W, Cfg::kTileH>(lt, L, (int)(((item + gridDim.x) / M) % lt.groups));
            compute_windows<TILE_W, Cfg::kTileH, Cfg::kSortSlots>(lt, L, tn, win[buf ^ 1], &win_slots[buf ^ 1], lane);
        }

        // ---- merge: equal slices of the record array, one per GW-lane group ----
        {
            // a group = GW lanes sharing a record; a lane owns NCH 16-byte chunks of the 128-byte rows.
            // GW = 4: chunk c0 = (lane & 3) | 4 * (group parity) and c0 ^ 4, so that the two halves of
            // the warp's groups read the two halves of the shared-memory banks
            constexpr int NCH = 8 / GW, kGroups = WARPS * (32 / GW);
            static_assert((Cfg::kRecs / kGroups) % 8 == 0, "slices are padded to multiples of 8 records");
            const int gl = lane / GW, cl = lane % GW;                  // group in warp, lane in group
            const int c0 = (GW == 8) ? cl : (cl | ((gl & 1) << 2));
            const int T = (int)(n_in + tail_ctr);
            // slice length: a multiple of 8 records (per * kGroups <= kRecs); what a slice holds beyond T
            // is filled with absent records by the group itself.  Slice of group gl of warp `warp`:
            // gl * WARPS + warp -- the sorted array runs from the coarsest level (long runs, few value
            // rows) to the finest and the unsorted rest, so every warp gets a slice of every part and
            // the warps finish together.
            const int per = (((T + kGroups - 1) / kGroups) + 7) & ~7;
            const int i0 = (gl * WARPS + warp) * per;
            for (int i = max(i0, T) + cl; i < i0 + per; i += GW) rec[i] = make_uint2(0xffffffffu, 0u);
            __syncwarp();
            // value / grad_value row of pixel 0 for this lane: + key * (M * 128) bytes per pixel (value rows:
            // M * 64 for 16-bit V); the lane's second chunk is the same address ^ 64 (value: ^ half a row).  Rows are
            // aligned to their size: host check
            const size_t lane_chunk = (size_t)(n * (long long)d.S * M + m) * 8 + c0;
            const char *v_lane = reinterpret_cast<const char *>(value) + lane_chunk * kChunkBytes<V>;
            char *gv_lane = reinterpret_cast<char *>(grad_value) + lane_chunk * 16;
            uint32_t row_bytes = (uint32_t)M * 128u;
            // keep the two 64-bit lane bases and the row stride as they are in registers: ptxas otherwise
            // splits them into a uniform and a per-lane part and re-adds / reloads them at every run start
            asm volatile("" : "+l"(v_lane), "+l"(gv_lane), "+r"(row_bytes));
            // value row stride: row_bytes for fp32, half of it for 16-bit V
            constexpr int kVShift = is16<V> ? 1 : 0;
            float4 acc[NCH];                                          // one 16-byte chunk each: leaves as one red.v4
            uint64_t v[2 * NCH];                                      // channel pairs: packed fp32x2 math
#pragma unroll
            for (int h = 0; h < NCH; ++h) acc[h] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int h = 0; h < 2 * NCH; ++h) v[h] = 0ull;
            constexpr uint32_t kNoKey = Cfg::kNoPix;       // shadows the 7-bit constant: this tile size's layout
            uint32_t cur = kNoKey;
            const uint32_t rec_s = smem_u32(rec) + (uint32_t)i0 * 8u;
            uint32_t go_s0 = smem_u32(go_sm) + (uint32_t)c0 * 16u, go_s1 = smem_u32(go_sm) + (uint32_t)(c0 ^ 4) * 16u;
            asm volatile("" : "+r"(go_s0), "+r"(go_s1));
            const uint32_t d_s = smem_u32(dsm);
            // The groups of a warp start at different bodies of their slices (and wrap around): slice
            // starts are multiples of 128 bytes apart, so walking them in step would put every group's
            // record reads on the same banks.  The wrap is just one more change of pixel.
            const int nb = per / GW;
            int bi = nb > 0 ? gl % nb : 0;
            for (int b = 0; b < nb; ++b) {
                const uint32_t ra = rec_s + (uint32_t)bi * (8u * GW);   // this body's GW records
                float dp[GW];
#pragma unroll
                for (int j = 0; j < GW; ++j) {
                    const uint2 rr = lds_u2(ra + 8u * j);
                    const uint32_t key = rr.x >> Cfg::kPixShift;
                    const uint32_t qoff = rr.x & Cfg::kQMask;                     // the query's grad_output row
                    uint64_t g[2 * NCH];
                    lds_2x64(go_s0 + qoff, g[0], g[1]);
                    if (NCH == 2) lds_2x64(go_s1 + qoff, g[2], g[3]);
                    if (key != cur) {                    // first record of a pixel (or of the padding)
                        if (cur != kNoKey) {
                            char *p = gv_lane + (size_t)cur * row_bytes;
                            red_add_f4(reinterpret_cast<float4 *>(p), acc[0]);
                            if (NCH == 2) red_add_f4(reinterpret_cast<float4 *>(xor64(p)), acc[NCH - 1]);
                        }
                        if (key != kNoKey) {
                            const char *p = v_lane + (size_t)key * (row_bytes >> kVShift);
                            ldg_value_chunk<V>(p, v[0], v[1]);
                            if (NCH == 2) ldg_value_chunk<V>(other_half<V>(p), v[2], v[3]);
                        }
                        cur = key;
#pragma unroll
                        for (int h = 0; h < NCH; ++h) {                          // the run's first term
                            fmul2_bcast_xy(acc[h].x, acc[h].y, rr.y, g[2 * h]);
                            fmul2_bcast_xy(acc[h].z, acc[h].w, rr.y, g[2 * h + 1]);
                        }
                    } else {
#pragma unroll
                        for (int h = 0; h < NCH; ++h) {                          // acc += weight * grad_output
                            ffma2_bcast_xy(acc[h].x, acc[h].y, rr.y, g[2 * h]);
                            ffma2_bcast_xy(acc[h].z, acc[h].w, rr.y, g[2 * h + 1]);
                        }
                    }
                    // <value row, grad_output row>: one packed dot product per 16-byte chunk, added at the
                    // end -- the sum does not depend on which chunk a lane happened to load first, so
                    // grad_sampling_loc / grad_attn_weight stay bit-reproducible from run to run
                    uint64_t d2 = 0ull, d2b = 0ull;
#pragma unroll
                    for (int h = 0; h < NCH; ++h) {
                        uint64_t t = fmul2_p(v[2 * h], g[2 * h]);
                        ffma2_p(t, v[2 * h + 1], g[2 * h + 1]);
                        if (h == 0) d2 = t; else d2b = t;
                    }
                    if (NCH == 2) d2 = fadd2_p(d2, d2b);
                    dp[j] = sum2(d2);
                }
                // D of record j: sum over the group's lanes; lane cl ends up with record j = cl
                float dsum;
                if (GW == 8) {
                    float r1[4], r2[2], r3[1];
                    rs_step<8>(reinterpret_cast<float (&)[8]>(dp), r1, cl & 4, 4);
                    rs_step<4>(r1, r2, cl & 2, 2);
                    rs_step<2>(r2, r3, cl & 1, 1);
                    dsum = r3[0];
                } else {
                    float r1[2], r2[1];
                    rs_step<4>(reinterpret_cast<float (&)[4]>(dp), r1, cl & 2, 2);
                    rs_step<2>(r1, r2, cl & 1, 1);
                    dsum = r2[0];
                }
                if (i0 + bi * GW + cl < T) {
                    const uint32_t xx = lds_u1(ra + 8u * (uint32_t)cl);
                    sts_f1(d_s + 4u * (((xx & Cfg::kQMask) >> 7) * (uint32_t)Cfg::kPC + (xx & 63u)), dsum);
                }
                if (++bi == nb) bi = 0;
            }
            if (cur != kNoKey) {
                char *p = gv_lane + (size_t)cur * row_bytes;
                red_add_f4(reinterpret_cast<float4 *>(p), acc[0]);
                if (NCH == 2) red_add_f4(reinterpret_cast<float4 *>(xor64(p)), acc[NCH - 1]);
            }
        }

        // ---- epilogue: grad_sampling_loc / grad_attn_weight, one point per thread ----
        // (the point is re-read from L2 rather than carried in registers across the merge loop; the
        // loads are issued before the barrier so that they fly while the warp waits)
        {
            const TileMap te = tile_of<TILE_W, Cfg::kTileH>(lt, L, g);
            Pair<PT> *gloc_n = reinterpret_cast<Pair<PT> *>(grad_loc) + n * Lq * (long long)M * LP;
            PT *gattw_n = grad_attw + n * Lq * (long long)M * LP;
            float2 exy[Cfg::kRounds];
            float2 erp[FUSED ? Cfg::kRounds : 1];
            float eaw[Cfg::kRounds];
            uint32_t erow[Cfg::kRounds];
            bool elive[Cfg::kRounds];
#pragma unroll
            for (int r = 0; r < Cfg::kRounds; ++r) {
                const int s = r * NT + tid;
                const int q = s / LP, p = s - q * LP;
                const int qg = s < Cfg::kPoints ? tile_query<TILE_W>(te, q, Lq) : -1;
                elive[r] = qg >= 0;
                erow[r] = (uint32_t)(qg * M + m) * (uint32_t)LP + (uint32_t)p;
                exy[r] = make_float2(0.f, 0.f);
                eaw[r] = 0.f;
                if (FUSED) erp[r] = make_float2(0.f, 0.f);
                if (elive[r]) {
                    exy[r] = ldg_stream_pair<PT>(loc_n + erow[r]);
                    if (FUSED)
                        erp[r] = ldg_stream_f2(reinterpret_cast<const float2 *>(
                            pr.ref + n * pr.ref_bstride + ((long long)qg * L + lt.level_of[p]) * 2));
                    else
                        eaw[r] = ldg_stream_one<PT>(attw_n + erow[r]);
                }
            }
            __syncthreads();                                                // B5: D complete
            float egx[Cfg::kRounds], egy[Cfg::kRounds], ega[Cfg::kRounds];
#pragma unroll
            for (int r = 0; r < Cfg::kRounds; ++r) {
                const int s = r * NT + tid;
                const int q = s / LP, p = s - q * LP;
                egx[r] = egy[r] = ega[r] = 0.f;
                if (elive[r]) {
                    const int l = lt.level_of[p];
                    const int4 lv = lt.hws[l];
                    float x = exy[r].x, y = exy[r].y, aw = eaw[r];
                    if (FUSED) {
                        const float2 rc = lt.rcp_wh[l];
                        x = erp[r].x + div_by_size(x, (float)lv.y, rc.x);
                        y = erp[r].y + div_by_size(y, (float)lv.x, rc.y);
                        aw = aw_sm[s];
                    }
                    const Geom<float> gm = decompose(x, y, lv.x, lv.y);
                    if (gm.cmask) {
                        const float4 D = reinterpret_cast<const float4 *>(dsm)[s];   // [q][p][corner]
                        const float d0 = (gm.cmask & 1) ? D.x : 0.f, d1 = (gm.cmask & 2) ? D.y : 0.f;
                        const float d2 = (gm.cmask & 4) ? D.z : 0.f, d3 = (gm.cmask & 8) ? D.w : 0.f;
                        const float lh = gm.lh, lw = gm.lw, hh = 1.f - gm.lh, hw = 1.f - gm.lw;
                        // cuh:161: sum_c grad_out[c] * val[c], val = w1 v1 + w2 v2 + w3 v3 + w4 v4
                        ega[r] = fmaf(hh * hw, d0, fmaf(hh * lw, d1, fmaf(lh * hw, d2, (lh * lw) * d3)));
                        // cuh:128-156,162-163: W * aw * sum_c g[c] (-hh v1 + hh v2 - lh v3 + lh v4), same for h
                        egx[r] = (aw * (float)lv.y) * fmaf(hh, d1 - d0, lh * (d3 - d2));
                        egy[r] = (aw * (float)lv.x) * fmaf(hw, d2 - d0, lw * (d3 - d1));
                    }
                    if (FUSED) {
                        // d location / d offset = 1 / (W, H) (mod.py:110-112)
                        egx[r] = __fdiv_rn(egx[r], (float)lv.y);
                        egy[r] = __fdiv_rn(egy[r], (float)lv.x);
                        scr_e[s] = aw * ega[r];                              // a_j * ga_j of this point
                    }
                }
            }
            if (FUSED) {
                __syncthreads();                                            // a_j * ga_j of the item visible
                // softmax backward: grad_logit_i = a_i * (ga_i - sum_j a_j ga_j) (torch: (grad - sum(grad * out)) * out)
#pragma unroll
                for (int r = 0; r < Cfg::kRounds; ++r) {
                    const int s = r * NT + tid;
                    if (elive[r]) {
                        const float *row = scr_e + (s / LP) * LP;
                        float dot = 0.f;
#pragma unroll
                        for (int j = 0; j < LP; ++j) dot += row[j];
                        ega[r] = aw_sm[s] * (ega[r] - dot);
                    }
                }
            }
#pragma unroll
            for (int r = 0; r < Cfg::kRounds; ++r) {
                if (elive[r]) {
                    stg_stream_pair<PT>(gloc_n + erow[r], egx[r], egy[r]);
                    stg_stream_v1<PT>(gattw_n + erow[r], ega[r]);
                }
            }
        }
    }
}

// ---------------------------------------------------------------------------
// host side: launch_bwd_sorted() serves the plain op and the fused producers (Producers::ref set),
// the latter in the default shapes only
// ---------------------------------------------------------------------------
template <typename V, int LP, int WARPS, int TILE_W, int MIN_CTAS, int TILE_Q, int SLOTS, int GW, bool FUSED>
static cudaError_t launch_bwd_sorted_cfg(const V *grad_out, const V *value, const int64_t *shapes,
                                         const int64_t *lstart, const ProducerT<V, FUSED> *loc,
                                         const ProducerT<V, FUSED> *attw, const Producers &pr, const Dims &d,
                                         float *gv, ProducerT<V, FUSED> *gl, ProducerT<V, FUSED> *gw, int gate,
                                         cudaStream_t stream) {
    using Cfg = SortCfg<LP, WARPS, TILE_W, TILE_Q, SLOTS>;
    constexpr auto kern = msda_bwd_sorted_kernel<V, LP, WARPS, TILE_W, MIN_CTAS, TILE_Q, SLOTS, GW, FUSED>;
    constexpr size_t kSmemBytes = Cfg::kSmem + (FUSED ? (size_t)Cfg::kPoints * sizeof(float) : 0);
    cudaError_t e;
    const int blocks = persistent_blocks<kern>(WARPS * 32, kSmemBytes, d, &e);
    if (blocks == 0) return e;
    const int flags = option_value(OPT_TILE_ORDER) != 1 ? 1 : 0;
    kern<<<blocks, WARPS * 32, kSmemBytes, stream>>>(grad_out, value, shapes, lstart, reinterpret_cast<const float *>(loc),
                                                     reinterpret_cast<const float *>(attw), pr, d, flags, gv,
                                                     reinterpret_cast<float *>(gl), reinterpret_cast<float *>(gw), gate);
    note_launch();
    return cudaGetLastError();
}

// whether launch_bwd_sorted() covers this problem (shape + alignment)
template <typename V>
bool bwd_sorted_applies(const V *value, const float *gv, const Dims &d) {
    // rows must be aligned to their size -- value: 32 * sizeof(V) bytes (128 fp32, 64 16-bit), grad_value (or the
    // 16-bit op's fp32 accumulation buffer): 128 -- because the merge loop addresses the two halves of a row as
    // p and p ^ (half a row); torch allocations are, odd views take the other kernel
    const bool rows_aligned = (reinterpret_cast<uintptr_t>(value) & (32u * sizeof(V) - 1u)) == 0 &&
                              (reinterpret_cast<uintptr_t>(gv) & 127u) == 0;
    return d32_applies(d) && d.Lq == d.S && (long long)d.S < (long long)kNoKey && rows_aligned;
}

// pr.ref == nullptr: plain; otherwise fused producers, gradients w.r.t. the raw sampling offsets (`loc`) and
// attention logits (`attw`), default shapes only (16-bit at L*P = 8: see below).  P: element type of `loc` / `attw` / `gl` / `gw` -- float, or V
// for the 16-bit fused producers.  `handled` = false: shape outside this kernel's domain (the caller falls back to
// msda_bwd.cu)
template <typename V, typename P>
cudaError_t launch_bwd_sorted(const V *grad_out, const V *value, const int64_t *shapes,
                              const int64_t *lstart, const P *loc, const P *attw, const Producers &pr,
                              const Dims &d, float *gv, P *gl, P *gw, int gate, cudaStream_t stream,
                              bool *handled) {
    *handled = bwd_sorted_applies(value, gv, d);
    if (!*handled) return cudaSuccess;
    // (warps, tile width, min CTAs per SM, queries per tile, window slots, lanes per record)
#define MSDA_SORTED(LPV, W, TW, C, TQ, SL, GWV, F) \
    launch_bwd_sorted_cfg<V, LPV, W, TW, C, TQ, SL, GWV, F>(grad_out, value, shapes, lstart, loc, attw, pr, d, gv, gl, \
                                                         gw, gate, stream)
    if constexpr (is16<P>) {   // 16-bit fused producers: 4 lanes per record, as fp32 fused (the same D summation order)
        switch (d.L * d.P) {
            case 4: return MSDA_SORTED(4, 16, 16, 2, 128, 4096, 4, true);
            // 8 warps, 64-query tiles, 3 CTAs per SM (85 registers): in the fp32 fused shape it spills
            case 8: return MSDA_SORTED(8, 8, 8, 3, 64, 2048, 4, true);
            case 12: return MSDA_SORTED(12, 16, 16, 2, 128, 4096, 4, true);
            default: return MSDA_SORTED(16, 16, 16, 1, 128, 4096, 4, true);
        }
    } else if constexpr (is16<V>) {   // 16-bit plain: the default shapes only
        switch (d.L * d.P) {
            case 4: return MSDA_SORTED(4, 16, 16, 2, 128, 4096, 8, false);
            case 8: return MSDA_SORTED(8, 16, 16, 2, 128, 4096, 8, false);
            case 12: return MSDA_SORTED(12, 16, 16, 2, 128, 4096, 4, false);
            default: return MSDA_SORTED(16, 16, 16, 1, 128, 4096, 8, false);
        }
    } else {
    if (pr.ref != nullptr) {
        switch (d.L * d.P) {   // 4, 8, 12 or 16 (d32_applies)
            case 4: return MSDA_SORTED(4, 16, 16, 2, 128, 4096, 4, true);
            case 8: return MSDA_SORTED(8, 16, 16, 2, 128, 4096, 4, true);
            case 12: return MSDA_SORTED(12, 16, 16, 2, 128, 4096, 4, true);
            default: return MSDA_SORTED(16, 16, 16, 1, 128, 4096, 4, true);
        }
    }
    const int variant = option_value(OPT_BWD_VARIANT);
    switch (d.L * d.P) {
        case 4: return MSDA_SORTED(4, 16, 16, 2, 128, 4096, 8, false);
        case 8: return MSDA_SORTED(8, 16, 16, 2, 128, 4096, 8, false);
        case 12:
            switch (variant) {      // tuning variants kept for tools/sweep.py (profiles/r2_sweep.md)
                case 21: return MSDA_SORTED(12, 16, 16, 2, 128, 4096, 8, false);   // 8 lanes per record (16 bytes each)
                case 24: return MSDA_SORTED(12, 12, 16, 2, 128, 4096, 4, false);   // 12 warps, 80 registers
                case 25: return MSDA_SORTED(12, 8, 8, 4, 64, 2048, 4, false);      // 64-query tiles, 4 CTAs of 8 warps
                case 27:
                    if (d.S < 0x1ffff) return MSDA_SORTED(12, 32, 16, 1, 256, 4096, 8, false);
                    return MSDA_SORTED(12, 16, 16, 2, 128, 4096, 4, false);
                case 26:                                                           // 256-query tiles (16 x 16), one CTA of 32 warps:
                    if (d.S < 0x1ffff) return MSDA_SORTED(12, 32, 16, 1, 256, 4096, 4, false);   // -2 % at configs[1], +2 % at 1024x2048
                    return MSDA_SORTED(12, 16, 16, 2, 128, 4096, 4, false);
                default: return MSDA_SORTED(12, 16, 16, 2, 128, 4096, 4, false);   // 128-query tiles, 2 CTAs of 16 warps, 4 lanes per record
            }
        default: return MSDA_SORTED(16, 16, 16, 1, 128, 4096, 8, false);
    }
    }
#undef MSDA_SORTED
}

#define MSDA_SORTED_V(V, P)                                                                                         \
    template cudaError_t launch_bwd_sorted<V, P>(const V *, const V *, const int64_t *, const int64_t *, const P *, \
                                                 const P *, const Producers &, const Dims &, float *, P *, P *, int, \
                                                 cudaStream_t, bool *);
template bool bwd_sorted_applies<float>(const float *, const float *, const Dims &);
template bool bwd_sorted_applies<__nv_bfloat16>(const __nv_bfloat16 *, const float *, const Dims &);
template bool bwd_sorted_applies<__half>(const __half *, const float *, const Dims &);
MSDA_SORTED_V(float, float)
MSDA_SORTED_V(__nv_bfloat16, float)
MSDA_SORTED_V(__half, float)
MSDA_SORTED_V(__nv_bfloat16, __nv_bfloat16)
MSDA_SORTED_V(__half, __half)
#undef MSDA_SORTED_V

}  // namespace msda
