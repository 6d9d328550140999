// linear_tf32x3.cu -- Y = X * W^T + bias (optionally ReLU) in fp32 on the sm_100a tensor cores.
//
// SURVEY.md 8f.3: once the MSDA op is fast, the pixel decoder's time is in its fp32 nn.Linear layers
// (value_proj / sampling_offsets / attention_weights / output_proj / FFN, msdeformattn.py:126-142,
// ops/modules/ms_deform_attn.py:62-65), which the reference runs as fp32 SIMT GEMMs (autocast is
// disabled, msdeformattn.py:338; TF32 matmuls are off by default in torch).  A plain TF32 GEMM would
// change the results (10-bit mantissa), so this kernel uses the error-compensated split
//     x = x_hi + x_lo,   x_hi = tf32(x),   x_lo = tf32(x - x_hi)
// (for X, x_hi = the upper 19 bits, which is what the tensor core reads from the raw fp32 tile)
//     X * W^T  ~=  Xhi*Whi^T + Xlo*Whi^T + Xhi*Wlo^T          (the dropped Xlo*Wlo^T term is ~2^-22)
// with fp32 accumulation in tensor memory: fp32-class accuracy at tensor-core speed.
//
// The tensor core adds each MMA's result into the fp32 accumulator with truncation (measured: the error
// of a single accumulator grows linearly with the number of MMAs), so the two small products go to a
// SECOND accumulator (2^-11 of the magnitude, hence 2^-11 of the truncation error) that is added in the
// epilogue: one third of the accumulations into the main one.
//
// Two kernels in this file (msda_b200_set_option("linear_variant", v) overrides the choice):
//   * linear_tf32x3_atmem_kernel -- the default: A operand (x_hi, x_lo) in tensor memory, see the comment
//     above it; reductions longer than 256 are accumulated in chunks of 256 that the epilogue warps add up
//     in registers (the truncating accumulation: error at the fp32 SIMT level needs few MMAs per accumulator);
//   * linear_tf32x3_kernel -- both operands in shared memory; with the weight split inside the kernel when no
//     workspace is given, and split-K (reductions into the zero-filled output) when the output has few tiles
//     and a very long reduction; with four accumulators {main, main', small, small'} it was the long-reduction
//     kernel before the chunked accumulation ("linear_variant" 2).
//
// Structure of linear_tf32x3_kernel (persistent: one CTA per SM walks 128 x BN output tiles, BN = 128 or 96;
// 14 warps):
//   pre-pass  W is split once per call into Whi / Wlo (workspace, 2 x N x K floats), unless WSPLIT;
//   warp 0   one thread: TMA loads of the fp32 X tile (128 x 32) and the Whi / Wlo tiles (BN x 32) of
//            each k-block into a STAGES-deep ring (128-byte swizzle: a tile row is one swizzle span);
//   warps 2-5 compute x_lo (and w_lo if WSPLIT) of the landed tiles element-wise into a second buffer (same
//            offsets -- the swizzle is irrelevant to an element-wise pass), fence to the async proxy and hand
//            the stage to
//   warp 1   one thread: the tcgen05.mma.kind::tf32 of the k-block (x_hi * [W_hi; W_lo]^T as ONE double-width
//            MMA into the adjacent {main, small} accumulators as soon as TMA has landed -- x_hi is the raw
//            tile --, x_lo * W_hi^T into small when the split is done), tcgen05.commit to release the stage;
//   warps 6-13 epilogue (of tile i while tile i+1 is computed when there are two accumulator sets):
//            tcgen05.ld the accumulators (lane = row) and add them up, hand the set back, then bias, ReLU,
//            32 x 32 transposes through shared memory and 128-byte row-segment stores (or reductions).
#include "tc_common.cuh"

#ifdef MSDA_PROFILE_KNOBS
// cycle counters of the pipeline roles (profiling build only; summed over the grid, see tools/whatif_linear_atmem.py)
__device__ unsigned long long g_lin_dbg[16];
#define LIN_DBG(...) __VA_ARGS__
#else
#define LIN_DBG(...)
#endif

namespace msda {

using namespace tc;

namespace {

constexpr int kSplitWarps = 4;    // warps 2-5
constexpr int kEpiWarps = 8;      // warps 6-13: two per TMEM lane quarter, alternating 32-column blocks
constexpr int kThreads = 64 + 32 * (kSplitWarps + kEpiWarps);
constexpr int kAccChunk = 8;      // k-blocks per accumulation chunk of the A-in-tensor-memory kernel

template <int BN, int STAGES, int NBUF, int NACC>
struct LinCfg {
    static constexpr int kXBytes = kBM * kBK * 4, kWBytes = BN * kBK * 4;
    static constexpr int kStageBytes = 2 * kXBytes + 2 * kWBytes;  // X hi, X lo, W hi, W lo
    static constexpr int kRingBytes = STAGES * kStageBytes;
    static constexpr int kEpiBytes = kEpiWarps * 32 * 33 * 4;      // 32 x 32 transpose tile (padded) per epilogue warp
    static constexpr int kSmem = kRingBytes + kEpiBytes + 1024 /* alignment slack */ + 256 /* barriers */;
    // NBUF accumulator sets (2: tile i is drained while tile i+1 is computed) of NACC accumulators of BN
    // columns: NACC == 2: {main, small}; NACC == 4: {main, main', small, small'} -- a tcgen05.mma that
    // accumulates into the result of the previous one waits ~240 cycles for it, so the products of a
    // k-step are spread over independent accumulators (the epilogue adds them up)
    static constexpr int kSetCols = NACC * BN;
    static constexpr int kTmemCols = NBUF * kSetCols <= 128 ? 128 : NBUF * kSetCols <= 256 ? 256 : 512;
    static_assert(NBUF * kSetCols <= 512 && BN % 32 == 0 && kStageBytes % 1024 == 0 && (NACC == 2 || NACC == 4), "tile shape");
};

// WSPLIT: W arrives as plain fp32 (map_wh) and is split inside the kernel like X -- for a one-shot "weight"
//         such as the transposed activations of a weight-gradient GEMM, where a pre-pass would cost a full
//         extra read and two writes of it.
// k_chunks > 1 (split-K): an output tile is computed by k_chunks CTAs-worth of work, each over kb_per_chunk
//         k-blocks, and added into y (zeroed by the launcher) with red.global.add -- for GEMMs with few
//         output tiles and a very long reduction (weight gradients: reduction over the rows).
//         ordered != 0 (deterministic entries): the launcher starts one CTA per output tile and the items are
//         numbered chunk-slowest, so CTA b walks the chunks of tile b in order; its epilogue stores chunk 0 and
//         adds every later chunk to what the same thread stored before -- the chunks' sums are added in chunk
//         order, with the accuracy of the chunked accumulation and without reductions in scheduling order.
template <int BN, int STAGES, int NBUF, int NACC, bool WSPLIT>
__global__ void __launch_bounds__(kThreads, 1)
linear_tf32x3_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_wh,
                     const __grid_constant__ CUtensorMap map_wl, const float *__restrict__ bias,
                     float *__restrict__ y, int M, int N, int K, int relu, int whatif, int k_chunks,
                     int kb_per_chunk, int ordered) {
    using Cfg = LinCfg<BN, STAGES, NBUF, NACC>;
    extern __shared__ uint8_t smem_dyn[];
    const uint32_t base = (smem_u32(smem_dyn) + 1023u) & ~1023u;         // 128-byte swizzle: 1024-byte aligned tiles
    uint8_t *base_ptr = smem_dyn + (base - smem_u32(smem_dyn));
    const uint32_t bars = base + Cfg::kRingBytes + Cfg::kEpiBytes;
    // ring barriers: full[s] (TMA landed), ready[s] (split done), empty[s] (MMAs done);
    // accumulator barriers: acc_full[b] (tile complete), acc_empty[b] (tile drained)
    auto full = [&](int s) { return bars + 8u * s; };
    auto ready = [&](int s) { return bars + 8u * (STAGES + s); };
    auto empty = [&](int s) { return bars + 8u * (2 * STAGES + s); };
    auto acc_full = [&](int b) { return bars + 8u * (3 * STAGES + b); };
    auto acc_empty = [&](int b) { return bars + 8u * (3 * STAGES + 2 + b); };
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(base_ptr + Cfg::kRingBytes + Cfg::kEpiBytes + 8 * (3 * STAGES + 4));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // timing experiments for profiles/ (results WRONG; msda_b200_set_option("whatif_linear", bits)):
    // 1 no MMAs, 2 no split work, 4 no output stores, 8 no W loads, 16 no X loads
    const bool dbg_no_mma = whatif & 1, dbg_no_split = whatif & 2, dbg_no_store = whatif & 4, dbg_no_w = whatif & 8,
               dbg_no_x = whatif & 16;
    const int kblocks_all = K / kBK;
    const int n_tiles = (N + BN - 1) / BN;
    // work items: (row block, column block, k chunk), chunk fastest (ordered: chunk slowest)
    const long long out_tiles = (long long)((M + kBM - 1) / kBM) * n_tiles;
    const long long tiles = out_tiles * k_chunks;
    // item -> (m0, n0, first k-block, number of k-blocks, rotation of the k order)
    auto decode = [&](long long t, int &m0, int &n0, int &kb0, int &nkb, int &rot) {
        const int chunk = ordered ? (int)(t / out_tiles) : (int)(t % k_chunks);
        const long long o = ordered ? t % out_tiles : t / k_chunks;
        m0 = (int)(o / n_tiles) * kBM;
        n0 = (int)(o % n_tiles) * BN;
        kb0 = chunk * kb_per_chunk;
        nkb = min(kb_per_chunk, kblocks_all - kb0);
        // every CTA starts its k loop at a different k-block: at any moment the SMs read different lines
        // of W (which all of them share) instead of queueing on the same L2 lines
        rot = (int)(blockIdx.x % (unsigned)nkb);
    };

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(full(s), 1);
            mbar_init(ready(s), 32 * kSplitWarps);
            mbar_init(empty(s), 1);
        }
        for (int b = 0; b < NBUF; ++b) {
            mbar_init(acc_full(b), 1);
            mbar_init(acc_empty(b), 32 * kEpiWarps);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     ::"r"(smem_u32(tmem_slot)), "r"(Cfg::kTmemCols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ---- TMA producer ----
        if (lane == 0) {
            uint32_t g = 0;                                               // k-blocks issued so far (ring position)
            for (long long t = blockIdx.x; t < tiles; t += gridDim.x) {
                int m0, n0, kb0, nkb, rot;
                decode(t, m0, n0, kb0, nkb, rot);
                for (int kb = 0; kb < nkb; ++kb, ++g) {
                    const int kk = kb0 + (kb + rot) % nkb;
                    const int s = g % STAGES;
                    mbar_wait(empty(s), ((g / STAGES) & 1) ^ 1);
                    const uint32_t st = base + s * Cfg::kStageBytes;
                    mbar_arrive_expect_tx(full(s), (dbg_no_x ? 0 : Cfg::kXBytes) + (dbg_no_w ? 0 : (WSPLIT ? 1 : 2) * Cfg::kWBytes));
                    if (!dbg_no_x) tma_load_2d(st, &map_x, full(s), kk * kBK, m0);
                    if (!dbg_no_w) tma_load_2d(st + 2 * Cfg::kXBytes, &map_wh, full(s), kk * kBK, n0);
                    if (!dbg_no_w && !WSPLIT) tma_load_2d(st + 2 * Cfg::kXBytes + Cfg::kWBytes, &map_wl, full(s), kk * kBK, n0);
                }
            }
        }
    } else if (warp == 1) {
        // ---- MMA issuer ----
        if (lane == 0) {
            constexpr uint32_t idesc = umma_idesc(kBM, BN), idesc2 = umma_idesc(kBM, 2 * BN > 256 ? BN : 2 * BN);
            uint32_t g = 0, it = 0;
            for (long long t = blockIdx.x; t < tiles; t += gridDim.x, ++it) {
                const uint32_t buf = it % NBUF;
                const uint32_t acc_set = tmem_base + buf * Cfg::kSetCols;
                mbar_wait(acc_empty(buf), ((it / NBUF) & 1) ^ 1);        // the epilogue has drained this set
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                int m0_, n0_, kb0_, nkb, rot_;
                decode(t, m0_, n0_, kb0_, nkb, rot_);
                for (int kb = 0; kb < nkb; ++kb, ++g) {
                    const int s = g % STAGES;
                    const uint32_t xh = base + s * Cfg::kStageBytes, xl = xh + Cfg::kXBytes;
                    const uint32_t wh = xl + Cfg::kXBytes, wl = wh + Cfg::kWBytes;
                    // the tensor core reads the upper 19 bits of an fp32 word as tf32, so the X tile as TMA
                    // delivered it IS x_hi = trunc(x): the two products that need only x_hi start at once ...
                    mbar_wait(full(s), (g / STAGES) & 1);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
                    for (int k = 0; k < kBK / kUmmaK; ++k) {
                        if (dbg_no_mma) continue;
                        const uint32_t ko = k * kUmmaK * 4;                // 32 bytes inside the swizzle span
                        if (NACC == 2) {
                            // {main, small} are adjacent in TMEM and W_hi, W_lo adjacent in the stage: ONE MMA of
                            // width 2*BN computes x_hi * [W_hi; W_lo]^T into both (x_hi is read once)
                            if (WSPLIT) {          // W_lo is not there yet: main product only
                                umma_tf32(acc_set, umma_desc(xh + ko), umma_desc(wh + ko), idesc, (kb | k) != 0);
                            } else {
                                umma_tf32(acc_set, umma_desc(xh + ko), umma_desc(wh + ko), idesc2, (kb | k) != 0);
                                if (2 * BN > 256) umma_tf32(acc_set + BN, umma_desc(xh + ko), umma_desc(wl + ko), idesc, (kb | k) != 0);
                            }
                        } else {                   // {main (even k-steps), main (odd), small: xl*wh, small: xh*wl}
                            umma_tf32(acc_set + (k & 1) * BN, umma_desc(xh + ko), umma_desc(wh + ko), idesc, (kb | (k >> 1)) != 0);
                            if (!WSPLIT) umma_tf32(acc_set + 3 * BN, umma_desc(xh + ko), umma_desc(wl + ko), idesc, (kb | k) != 0);
                        }
                    }
                    // ... and x_lo * w_hi follows when the split warps have produced x_lo
                    mbar_wait(ready(s), (g / STAGES) & 1);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
                    for (int k = 0; k < kBK / kUmmaK; ++k) {
                        if (dbg_no_mma) continue;
                        const uint32_t ko = k * kUmmaK * 4;
                        if (NACC == 2) {
                            if (WSPLIT) umma_tf32(acc_set + BN, umma_desc(xh + ko), umma_desc(wl + ko), idesc, (kb | k) != 0);
                            umma_tf32(acc_set + BN, umma_desc(xl + ko), umma_desc(wh + ko), idesc, 1);
                        } else {
                            if (WSPLIT) umma_tf32(acc_set + 3 * BN, umma_desc(xh + ko), umma_desc(wl + ko), idesc, (kb | k) != 0);
                            umma_tf32(acc_set + 2 * BN, umma_desc(xl + ko), umma_desc(wh + ko), idesc, (kb | k) != 0);
                        }
                    }
                    umma_commit(empty(s));                                // stage reusable once these MMAs are done
                }
                umma_commit(acc_full(buf));
            }
        }
    } else if (warp < 2 + kSplitWarps) {
        // ---- split warps: x_lo = tf32(x - trunc19(x)) ----
        const int t0 = threadIdx.x - 64;
        uint32_t g = 0;
        for (long long t = blockIdx.x; t < tiles; t += gridDim.x) {
            int m0_, n0_, kb0_, nkb, rot_;
            decode(t, m0_, n0_, kb0_, nkb, rot_);
            for (int kb = 0; kb < nkb; ++kb, ++g) {
                const int s = g % STAGES;
                mbar_wait(full(s), (g / STAGES) & 1);
                // the stage is [X | X_lo | W_hi | W_lo]; lo = tf32(v - trunc19(v)) goes kXBytes (X) or kWBytes (W) further
                float4 *stage4 = reinterpret_cast<float4 *>(base_ptr + s * Cfg::kStageBytes);
                constexpr int kX4 = Cfg::kXBytes / 16, kW4 = Cfg::kWBytes / 16;
#pragma unroll
                for (int c = t0; c < (dbg_no_split ? 0 : kX4 + (WSPLIT ? kW4 : 0)); c += 32 * kSplitWarps) {
                    const bool is_w = WSPLIT && c >= kX4;
                    const int src = is_w ? c + kX4 : c;                   // W_hi starts 2 * kX4 into the stage
                    const int dst = src + (is_w ? kW4 : kX4);
                    const float4 v = stage4[src];
                    uint4 l;
                    l.x = to_tf32(v.x - __uint_as_float(__float_as_uint(v.x) & 0xffffe000u));
                    l.y = to_tf32(v.y - __uint_as_float(__float_as_uint(v.y) & 0xffffe000u));
                    l.z = to_tf32(v.z - __uint_as_float(__float_as_uint(v.z) & 0xffffe000u));
                    l.w = to_tf32(v.w - __uint_as_float(__float_as_uint(v.w) & 0xffffe000u));
                    *reinterpret_cast<uint4 *>(stage4 + dst) = l;
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes -> tensor core reads
                mbar_arrive(ready(s));
            }
        }
    } else {
        // ---- epilogue warps: TMEM lane = row; warp w may touch lanes 32*(w%4) .. +31 ----
        const int q = warp & 3;
        float *tile = reinterpret_cast<float *>(base_ptr + Cfg::kRingBytes) + (warp - 2 - kSplitWarps) * 32 * 33;
        uint32_t it = 0;
        for (long long t = blockIdx.x; t < tiles; t += gridDim.x, ++it) {
            int m0, n0, kb0, nkb_, rot_;
            decode(t, m0, n0, kb0, nkb_, rot_);
            const uint32_t buf = it % NBUF;
            const uint32_t acc = tmem_base + buf * Cfg::kSetCols + ((uint32_t)(q * 32) << 16);
            mbar_wait(acc_full(buf), (it / NBUF) & 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            // this warp's 32-column blocks: c = part, part + kEpiWarps/4, ...  All of them are read from TMEM and
            // their accumulators added up before anything else, so the set goes back to the MMA warp after a few
            // hundred cycles; the transposes and stores then overlap with the MMAs of the next tile
            constexpr int kStep = kEpiWarps / 4, kMaxBlk = (BN / 32 + kStep - 1) / kStep;
            const int part = (warp - 2 - kSplitWarps) >> 2;
            float sum[kMaxBlk][32];
#pragma unroll
            for (int i = 0; i < kMaxBlk; ++i) {
                const int c = part + i * kStep;
                if (c < BN / 32) {
                    uint32_t v[32], u[32];
                    tmem_ld32(acc + (uint32_t)(c * 32), v);
                    tmem_ld32(acc + (uint32_t)(BN + c * 32), u);
#pragma unroll
                    for (int j = 0; j < 32; ++j) sum[i][j] = __uint_as_float(v[j]) + __uint_as_float(u[j]);
                    if (NACC == 4) {                                      // (main + main') + (small + small')
                        tmem_ld32(acc + (uint32_t)(2 * BN + c * 32), v);
                        tmem_ld32(acc + (uint32_t)(3 * BN + c * 32), u);
#pragma unroll
                        for (int j = 0; j < 32; ++j) sum[i][j] += __uint_as_float(v[j]) + __uint_as_float(u[j]);
                    }
                }
            }
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            mbar_arrive(acc_empty(buf));
#pragma unroll
            for (int i = 0; i < kMaxBlk; ++i) {
                const int c = part + i * kStep;
                if (c >= BN / 32) continue;
                const int col = n0 + c * 32;
                const float b = (bias != nullptr && col + lane < N && kb0 == 0) ? bias[col + lane] : 0.f;
#pragma unroll
                for (int j = 0; j < 32; ++j) tile[lane * 33 + j] = sum[i][j];
                __syncwarp();
                if (k_chunks == 1) {               // (kept apart from the split-K loop: an asm with a memory clobber in
#pragma unroll 8                                   //  the body stops the compiler from batching the shared loads)
                    for (int r = 0; r < 32; ++r) {
                        const int row = m0 + q * 32 + r;
                        float o = tile[r * 33 + lane] + b;
                        if (relu) o = fmaxf(o, 0.f);
                        if (row < M && col + lane < N && !dbg_no_store) y[(long long)row * N + col + lane] = o;
                    }
                } else if (ordered) {              // this thread stored the tile's earlier chunks of these elements
#pragma unroll 8
                    for (int r = 0; r < 32; ++r) {
                        const int row = m0 + q * 32 + r;
                        const float o = tile[r * 33 + lane] + b;
                        if (row < M && col + lane < N) {
                            float *p = y + (long long)row * N + col + lane;
                            *p = kb0 == 0 ? o : *p + o;
                        }
                    }
                } else {
#pragma unroll 8
                    for (int r = 0; r < 32; ++r) {
                        const int row = m0 + q * 32 + r;
                        const float o = tile[r * 33 + lane] + b;
                        if (row < M && col + lane < N)
                            asm volatile("red.global.add.f32 [%0], %1;" ::"l"(y + (long long)row * N + col + lane), "f"(o));
                    }
                }
                __syncwarp();
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(Cfg::kTmemCols) : "memory");
}

// ---------------------------------------------------------------------------
// Kernel with the A operand in tensor memory (the default).  With both operands in shared memory a
// 128 x 128 x 8 tf32 MMA reads 8 KB for 64 cycles of math and the shared-memory data pipe is the limit
// (profiles/r1_linear.md).  Here the split warps write x_hi (the raw words) and x_lo of their 32 rows into a
// 4-slot ring in TMEM with tcgen05.st (lane = row, 32 columns = the 32 k of a k-block) and the MMAs take A
// from there ([tmem] operand form): operand reads from shared memory are halved and x_lo is never stored
// to shared memory.  TMEM: {main, small} accumulators (2 * BN columns, one set: the epilogue warps drain it
// into registers at once and hand it back, their transposes and stores overlap the next tile's MMAs) +
// 4 x 64 columns of A.  Epilogue buffer: 32 x 32 floats per warp, XOR-swizzled 16-byte chunks (kEpiBytes
// keeps round 1's padded size).
// ---------------------------------------------------------------------------
template <int BN>
struct LinCfgT {
    static constexpr int kStages = 4;
    static constexpr int kXBytes = kBM * kBK * 4, kWBytes = BN * kBK * 4;
    static constexpr int kStageBytes = kXBytes + 2 * kWBytes;      // X (raw), W hi, W lo
    static constexpr int kRingBytes = kStages * kStageBytes;
    static constexpr int kEpiBytes = kEpiWarps * 32 * 33 * 4;
    static constexpr int kSmem = kRingBytes + kEpiBytes + 1024 + 256;
    static constexpr int kACol = 2 * BN;                           // first TMEM column of the A ring
    static constexpr int kTmemCols = 512;
    static_assert(2 * BN + kStages * 64 <= 512 && kStageBytes % 1024 == 0, "tile shape");
};

template <int BN>
__global__ void __launch_bounds__(kThreads, 1)
linear_tf32x3_atmem_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_wh,
                           const __grid_constant__ CUtensorMap map_wl, const float *__restrict__ bias,
                           float *__restrict__ y, int M, int N, int K, int relu, int kb_chunk, int whatif) {
    using Cfg = LinCfgT<BN>;
    // timing experiments for profiles/ (results WRONG; profiling build only, msda_b200_set_option("whatif_linear", bits);
    // compile-time false in the shipped library)
#ifdef MSDA_PROFILE_KNOBS
    const bool dbg_no_mma2 = whatif & 1, dbg_no_split = whatif & 2, dbg_no_store = whatif & 4, dbg_no_mma1 = whatif & 8,
               dbg_narrow = whatif & 16, dbg_alt = whatif & 32, dbg_no_wlo = whatif & 64, dbg_no_w = whatif & 128, dbg_no_x = whatif & 256,
               dbg_no_sttm = whatif & 512, dbg_no_lds = whatif & 1024, dbg_plain_arrive = whatif & 2048,
               dbg_no_epi = whatif & 4096, dbg_poll = whatif & 8192;
#else
    constexpr bool dbg_no_mma2 = false, dbg_no_split = false, dbg_no_store = false, dbg_no_mma1 = false, dbg_narrow = false,
                   dbg_alt = false, dbg_no_wlo = false, dbg_no_w = false, dbg_no_x = false, dbg_no_sttm = false,
                   dbg_no_lds = false, dbg_plain_arrive = false, dbg_no_epi = false, dbg_poll = false;
    (void)whatif;
#endif
    auto WAIT = [&](uint32_t bar, uint32_t parity) { if (dbg_poll) mbar_wait_poll(bar, parity); else mbar_wait(bar, parity); };
    constexpr int STAGES = Cfg::kStages;
    extern __shared__ uint8_t smem_dyn[];
    const uint32_t base = (smem_u32(smem_dyn) + 1023u) & ~1023u;
    uint8_t *base_ptr = smem_dyn + (base - smem_u32(smem_dyn));
    const uint32_t bars = base + Cfg::kRingBytes + Cfg::kEpiBytes;
    auto full = [&](int s) { return bars + 8u * s; };
    auto ready = [&](int s) { return bars + 8u * (STAGES + s); };
    auto empty = [&](int s) { return bars + 8u * (2 * STAGES + s); };
    const uint32_t acc_full = bars + 8u * 3 * STAGES, acc_empty = acc_full + 8u;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(base_ptr + Cfg::kRingBytes + Cfg::kEpiBytes + 8 * (3 * STAGES + 2));

    // the warp index through a shuffle: the compiler then KNOWS it is warp-uniform and keeps the role loops' addresses
    // and descriptors in uniform registers
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    LIN_DBG(__shared__ volatile long long ts_issue[Cfg::kStages]; __shared__ volatile long long ts_commit[Cfg::kStages];
            long long d0 = 0, d1 = 0, d2 = 0, d3 = 0; const long long t_start = clock64();)
    const int kblocks = K / kBK;
    const int n_tiles = (N + BN - 1) / BN;
    const long long tiles = (long long)((M + kBM - 1) / kBM) * n_tiles;

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(full(s), 1);
            mbar_init(ready(s), kSplitWarps);               // one arrival per warp (lane 0, after __syncwarp)
            mbar_init(empty(s), 1);
        }
        mbar_init(acc_full, 1);
        mbar_init(acc_empty, kEpiWarps);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     ::"r"(smem_u32(tmem_slot)), "r"(Cfg::kTmemCols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);

    if (warp == 0) {
        if (lane == 0) {
            uint32_t g = 0;
            for (long long t = blockIdx.x; t < tiles; t += gridDim.x) {
                const int m0 = (int)(t / n_tiles) * kBM, n0 = (int)(t % n_tiles) * BN;
                for (int kb = 0; kb < kblocks; ++kb, ++g) {
                    const int kk = kb;      // the same k order for every tile: a row's result does not depend on which
                                            // CTA computed it (row-range sharding reproduces the unsharded bits)
                    const int s = g % STAGES;
                    LIN_DBG(const long long w0 = clock64();)
                    WAIT(empty(s), ((g / STAGES) & 1) ^ 1);
                    LIN_DBG(const long long w1 = clock64(); d0 += w1 - w0; d1 += 1; if (g >= STAGES) d2 += w1 - ts_commit[s]; ts_issue[s] = w1;)
                    const uint32_t st = base + s * Cfg::kStageBytes;
                    mbar_arrive_expect_tx(full(s), Cfg::kStageBytes - (dbg_no_w ? 2 : dbg_no_wlo ? 1 : 0) * Cfg::kWBytes -
                                                       (dbg_no_x ? Cfg::kXBytes : 0));
                    if (!dbg_no_x) tma_load_2d(st, &map_x, full(s), kk * kBK, m0);
                    if (!dbg_no_w) tma_load_2d(st + Cfg::kXBytes, &map_wh, full(s), kk * kBK, n0);
                    if (!dbg_no_w && !dbg_no_wlo) tma_load_2d(st + Cfg::kXBytes + Cfg::kWBytes, &map_wl, full(s), kk * kBK, n0);
                }
            }
            LIN_DBG(atomicAdd(&g_lin_dbg[0], d0); atomicAdd(&g_lin_dbg[1], d1); atomicAdd(&g_lin_dbg[12], d2);)
        }
    } else if (warp == 1) {
        // The whole warp walks the loop (warp-uniform control flow, everything in uniform registers); one elected lane
        // issues.  A tcgen05.mma is accepted only when the previous one is nearly done (measured: the issue of a
        // k-block's 8 MMAs takes their execution time), so every instruction BETWEEN two issues is tensor-core idle
        // time: the descriptors of a k-block differ from the stage's first one by constants.
        constexpr uint32_t idesc = umma_idesc(kBM, BN), idesc2 = umma_idesc(kBM, 2 * BN);
        const bool leader = elect_one();
        uint32_t g = 0, it = 0;                                           // it: accumulation chunks so far
        LIN_DBG(long long w3 = 0;)
        for (long long t = blockIdx.x; t < tiles; t += gridDim.x) {
            int kc = 0;                                                    // position in the accumulation chunk
            for (int kb = 0; kb < kblocks; ++kb, ++g) {
                if (kc == 0) {
                    LIN_DBG(const long long w0 = clock64();)
                    WAIT(acc_empty, (it & 1) ^ 1);
                    LIN_DBG(d2 += clock64() - w0;)
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                }
                const int s = g % STAGES;
                LIN_DBG(const long long w2 = clock64();)
                WAIT(ready(s), (g / STAGES) & 1);                          // A slot written (implies the W tiles landed)
                LIN_DBG(w3 = clock64(); d0 += w3 - w2;)
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint64_t dw = umma_desc(base + s * Cfg::kStageBytes + Cfg::kXBytes);
                const uint32_t a_hi = tmem_base + Cfg::kACol + s * 64, a_lo = a_hi + 32;
                if (leader) {
#pragma unroll
                    for (int k = 0; k < kBK / kUmmaK; ++k) {
                        const uint64_t db = dw + (uint64_t)((k * kUmmaK * 4) >> 4);   // + 32 bytes per k-step (address field, no carry)
                        // x_hi * [W_hi; W_lo]^T -> {main, small};  x_lo * W_hi^T -> small
                        if (!dbg_no_mma1)
                            umma_tf32_ts(tmem_base, a_hi + k * kUmmaK, db, dbg_narrow ? idesc : idesc2, (kc | k) != 0);
                        if (!dbg_no_mma2)     // dbg_alt: into the main accumulator (no dependence on the double-width MMA's small half)
                            umma_tf32_ts(tmem_base + (dbg_alt ? 0 : BN), a_lo + k * kUmmaK, db, idesc, 1);
                    }
                    if (dbg_plain_arrive) mbar_arrive(empty(s)); else
                    umma_commit(empty(s));                                 // smem stage AND TMEM A slot reusable
                }
                LIN_DBG(const long long w4 = clock64(); d1 += w4 - w3; if (leader) ts_commit[s] = w4;)
                if (++kc == kb_chunk || kb == kblocks - 1) {
                    if (leader) {
                        if (dbg_plain_arrive) mbar_arrive(acc_full); else
                        umma_commit(acc_full);                             // this chunk's sums are complete
                    }
                    ++it;
                    kc = 0;
                }
            }
        }
        LIN_DBG(if (leader) { atomicAdd(&g_lin_dbg[5], d0); atomicAdd(&g_lin_dbg[6], d1); atomicAdd(&g_lin_dbg[7], d2); })
    } else if (warp < 2 + kSplitWarps) {
        // ---- A warps: rows 32*(warp%4) .. +31 of the X tile -> TMEM (x_hi = raw words, x_lo) ----
        // (two warps per lane quarter on alternate k-blocks were tried: the 576-thread CTA's 96-register cap
        //  spills the epilogue, 0.218 -> 0.242 ms at 256 x 256)
        const int q = warp & 3, row = q * 32 + lane;
        uint32_t g = 0;
        for (long long t = blockIdx.x; t < tiles; t += gridDim.x) {
            for (int kb = 0; kb < kblocks; ++kb, ++g) {
                const int s = g % STAGES;
                LIN_DBG(const long long w0 = clock64();)
                WAIT(full(s), (g / STAGES) & 1);
                LIN_DBG(const long long w1 = clock64(); d0 += w1 - w0; d2 += w1 - ts_issue[s];)
                const uint8_t *xrow = base_ptr + s * Cfg::kStageBytes + row * 128;
                uint32_t hi[32], lo[32];
#pragma unroll
                for (int j = 0; j < 8; ++j) {                              // 128-byte swizzle: chunk j sits at j ^ (row % 8)
                    const uint4 v = dbg_no_lds ? make_uint4(j, g, s, row) : *reinterpret_cast<const uint4 *>(xrow + ((j ^ (row & 7)) << 4));
                    hi[4 * j + 0] = v.x; hi[4 * j + 1] = v.y; hi[4 * j + 2] = v.z; hi[4 * j + 3] = v.w;
                }
#pragma unroll
                for (int j = 0; j < 32; ++j)
                    lo[j] = dbg_no_split ? hi[j] : to_tf32(__uint_as_float(hi[j]) - __uint_as_float(hi[j] & 0xffffe000u));
                const uint32_t a_hi = tmem_base + ((uint32_t)(q * 32) << 16) + Cfg::kACol + s * 64;
                if (!dbg_no_sttm) {
                    tmem_st32(a_hi, hi);
                    tmem_st32(a_hi + 32, lo);
                    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
                } else if (hi[3] == 0x12345u && lo[7] == 0x54321u) {
                    y[0] = 1.f;                                            // keeps the loads and the split alive
                }
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                __syncwarp();
                if (lane == 0) mbar_arrive(ready(s));
                LIN_DBG(d1 += clock64() - w1;)
            }
        }
        LIN_DBG(if (warp == 2 && lane == 0) { atomicAdd(&g_lin_dbg[2], d0); atomicAdd(&g_lin_dbg[3], d1); atomicAdd(&g_lin_dbg[4], d2); })
    } else {
        const int q = warp & 3;
        float4 *tile4 = reinterpret_cast<float4 *>(base_ptr + Cfg::kRingBytes) + (warp - 2 - kSplitWarps) * 32 * 8;
        uint32_t it = 0;                                                  // accumulation chunks so far
        for (long long t = blockIdx.x; t < tiles; t += gridDim.x) {
            const int m0 = (int)(t / n_tiles) * kBM, n0 = (int)(t % n_tiles) * BN;
            const uint32_t acc = tmem_base + ((uint32_t)(q * 32) << 16);
            // this warp's 32-column blocks: c = part, part + kEpiWarps/4, ...  All of them are read from TMEM
            // (and main + small added) before anything else, so the accumulators go back to the MMA warp after
            // a few hundred cycles; the transposes and stores then overlap with the next tile's MMAs
            constexpr int kStep = kEpiWarps / 4, kMaxBlk = (BN / 32 + kStep - 1) / kStep;
            const int part = (warp - 2 - kSplitWarps) >> 2;
            float sum[kMaxBlk][32];
            // long reductions are accumulated in chunks of kb_chunk k-blocks: the tensor core adds every MMA
            // into the accumulator with truncation, so the error of one accumulator grows with its number of
            // MMAs; each chunk starts from fresh accumulators and the chunks are added here in fp32 registers
            // (round to nearest) -- the error stays at the level of a 256-deep reduction
#pragma unroll
            for (int i = 0; i < kMaxBlk; ++i)
#pragma unroll
                for (int j = 0; j < 32; ++j) sum[i][j] = 0.f;
            LIN_DBG(d3 = clock64();)
            for (int kb0 = 0; kb0 < kblocks; kb0 += kb_chunk, ++it) {
                LIN_DBG(const long long w0 = clock64();)
                WAIT(acc_full, it & 1);
                LIN_DBG(const long long w1 = clock64(); d0 += w1 - w0;)
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
                for (int i = 0; i < kMaxBlk; ++i) {
                    const int c = part + i * kStep;
                    if (c < BN / 32) {
                        uint32_t v[32];                                    // main, then small
                        tmem_ld32(acc + (uint32_t)(c * 32), v);
#pragma unroll
                        for (int j = 0; j < 32; ++j) sum[i][j] += __uint_as_float(v[j]);
                        tmem_ld32(acc + (uint32_t)(BN + c * 32), v);
#pragma unroll
                        for (int j = 0; j < 32; ++j) sum[i][j] += __uint_as_float(v[j]);
                    }
                }
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                __syncwarp();
                if (lane == 0) mbar_arrive(acc_empty);
                LIN_DBG(d3 = clock64(); d1 += d3 - w1;)
            }
            // 32 x 32 blocks go through shared memory to turn "lane = row" into row segments: 128-bit accesses both
            // ways, chunk c of row r at position c ^ (r % 8) (no padding, no bank conflicts), then one 128-bit global
            // store per lane = four 128-byte row segments per instruction -- a quarter of the instructions of a
            // scalar loop, which matters beyond the epilogue: these warps share issue slots with the single thread
            // that feeds the tensor core
            const int sub = lane >> 3, ch = lane & 7;                    // row within a group of 4, 16-byte chunk
#pragma unroll
            for (int i = 0; i < kMaxBlk; ++i) {
                const int c = part + i * kStep;
                if (c >= BN / 32 || dbg_no_epi) continue;
                const int col = n0 + c * 32 + ch * 4;                     // this lane's 4 columns in the store loop
                float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
                if (bias != nullptr && col < N) b4 = make_float4(bias[col], bias[col + 1], bias[col + 2], bias[col + 3]);
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    tile4[lane * 8 + (j ^ (lane & 7))] = make_float4(sum[i][4 * j], sum[i][4 * j + 1], sum[i][4 * j + 2], sum[i][4 * j + 3]);
                __syncwarp();
                float *yrow = y + (long long)(m0 + q * 32 + sub) * N + col;
#pragma unroll
                for (int r4 = 0; r4 < 8; ++r4) {
                    const int r = r4 * 4 + sub;
                    float4 o = tile4[r * 8 + (ch ^ (r & 7))];
                    o.x += b4.x; o.y += b4.y; o.z += b4.z; o.w += b4.w;
                    if (relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
                    if (m0 + q * 32 + r < M && col < N && !dbg_no_store)
                        *reinterpret_cast<float4 *>(yrow + (long long)r4 * 4 * N) = o;
                }
                __syncwarp();
            }
            LIN_DBG(d2 += clock64() - d3;)
        }
        LIN_DBG(if (warp == 2 + kSplitWarps && lane == 0) { atomicAdd(&g_lin_dbg[8], d0); atomicAdd(&g_lin_dbg[9], d1); atomicAdd(&g_lin_dbg[10], d2); })
    }
    LIN_DBG(if (threadIdx.x == 0) atomicAdd(&g_lin_dbg[11], clock64() - t_start);)
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(Cfg::kTmemCols) : "memory");
}

// W -> (tf32(W), tf32(W - tf32(W))), once per call
__global__ void split_weight_kernel(const float4 *__restrict__ w, float4 *__restrict__ hi, float4 *__restrict__ lo, long long n4) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
        const float4 v = w[i];
        uint4 h, l;
        h.x = to_tf32(v.x); h.y = to_tf32(v.y); h.z = to_tf32(v.z); h.w = to_tf32(v.w);
        l.x = to_tf32(v.x - __uint_as_float(h.x));
        l.y = to_tf32(v.y - __uint_as_float(h.y));
        l.z = to_tf32(v.z - __uint_as_float(h.z));
        l.w = to_tf32(v.w - __uint_as_float(h.w));
        reinterpret_cast<uint4 *>(hi)[i] = h;
        reinterpret_cast<uint4 *>(lo)[i] = l;
    }
}

// ---- host side ----
template <int BN, int STAGES, int NBUF, int NACC, bool WSPLIT>
cudaError_t launch_linear(const float *x, const float *w, const float *bias, float *y, int M, int N, int K,
                          int relu, float *workspace, cudaStream_t stream, bool deterministic) {
    using Cfg = LinCfg<BN, STAGES, NBUF, NACC>;
    auto kern = linear_tf32x3_kernel<BN, STAGES, NBUF, NACC, WSPLIT>;
    static std::atomic<bool> attr_set[msda::kMaxDevices];
    {
        cudaError_t e = cudaSuccess;
        const int dev = msda::device_slot(&e);
        if (dev < 0) return e;
        if (!attr_set[dev].load(std::memory_order_acquire)) {
            e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmem);
            if (e != cudaSuccess) return e;
            attr_set[dev].store(true, std::memory_order_release);
        }
    }
    CUtensorMap mx, mwh, mwl;
    if (WSPLIT) {
        if (!make_map(&mx, x, M, K, kBM) || !make_map(&mwh, w, N, K, BN)) return cudaErrorInvalidValue;
        mwl = mwh;
    } else {
        float *whi = workspace, *wlo = workspace + (size_t)N * K;
        if (!make_map(&mx, x, M, K, kBM) || !make_map(&mwh, whi, N, K, BN) || !make_map(&mwl, wlo, N, K, BN))
            return cudaErrorInvalidValue;
        const long long n4 = (long long)N * K / 4;
        split_weight_kernel<<<(unsigned)((n4 + 255) / 256 < 592 ? (n4 + 255) / 256 : 592), 256, 0, stream>>>(
            reinterpret_cast<const float4 *>(w), reinterpret_cast<float4 *>(whi), reinterpret_cast<float4 *>(wlo), n4);
        note_launch();
    }
    // split-K when the output has too few tiles to occupy the GPU and the reduction is long (deterministic
    // entries: the same chunks, walked in order by one CTA per tile, see the kernel)
    const long long out_tiles = (long long)((M + kBM - 1) / kBM) * ((N + BN - 1) / BN);
    const int kblocks = K / kBK;
    int k_chunks = 1;
    if (out_tiles * 2 <= sm_count() && kblocks >= 64 && !relu) {
        const long long want = (2LL * sm_count() + out_tiles - 1) / out_tiles;    // ~2 work items per SM
        k_chunks = (int)(want < kblocks / 16 ? want : kblocks / 16);
        if (k_chunks < 1) k_chunks = 1;
    }
    const int kb_per_chunk = (kblocks + k_chunks - 1) / k_chunks;
    k_chunks = (kblocks + kb_per_chunk - 1) / kb_per_chunk;
    const int ordered = deterministic && k_chunks > 1;
    if (k_chunks > 1 && !ordered) {
        cudaError_t e = cudaMemsetAsync(y, 0, (size_t)M * N * sizeof(float), stream);
        if (e != cudaSuccess) return e;
    }
    const long long tiles = out_tiles * k_chunks;
    // persistent: one CTA per SM; ordered: one CTA per output tile (out_tiles * 2 <= SMs here)
    const long long grid = ordered ? out_tiles : (tiles < sm_count() ? tiles : sm_count());
    kern<<<(unsigned)grid, kThreads, Cfg::kSmem, stream>>>(mx, mwh, mwl, bias, y, M, N, K, relu,
                                                           whatif_value(OPT_WHATIF_LINEAR), k_chunks, kb_per_chunk,
                                                           ordered);
    note_launch();
    return cudaGetLastError();
}

template <int BN>
cudaError_t launch_linear_atmem(const float *x, const float *w, const float *bias, float *y, int M, int N, int K,
                                int relu, float *workspace, cudaStream_t stream) {
    using Cfg = LinCfgT<BN>;
    auto kern = linear_tf32x3_atmem_kernel<BN>;
    static std::atomic<bool> attr_set[msda::kMaxDevices];
    {
        cudaError_t e = cudaSuccess;
        const int dev = msda::device_slot(&e);
        if (dev < 0) return e;
        if (!attr_set[dev].load(std::memory_order_acquire)) {
            e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmem);
            if (e != cudaSuccess) return e;
            attr_set[dev].store(true, std::memory_order_release);
        }
    }
    float *whi = workspace, *wlo = workspace + (size_t)N * K;
    CUtensorMap mx, mwh, mwl;
    if (!make_map(&mx, x, M, K, kBM) || !make_map(&mwh, whi, N, K, BN) || !make_map(&mwl, wlo, N, K, BN))
        return cudaErrorInvalidValue;
    if (w != nullptr) {              // nullptr: the workspace already holds the split weight (launch_split_weight)
        const long long n4 = (long long)N * K / 4;
        split_weight_kernel<<<(unsigned)((n4 + 255) / 256 < 592 ? (n4 + 255) / 256 : 592), 256, 0, stream>>>(
            reinterpret_cast<const float4 *>(w), reinterpret_cast<float4 *>(whi), reinterpret_cast<float4 *>(wlo), n4);
        note_launch();
    }
    const long long tiles = (long long)((M + kBM - 1) / kBM) * ((N + BN - 1) / BN);
    const long long grid = tiles < sm_count() ? tiles : sm_count();
    // accumulation chunks of 8 k-blocks (256 of the reduction) -- see the epilogue
    kern<<<(unsigned)grid, kThreads, Cfg::kSmem, stream>>>(mx, mwh, mwl, bias, y, M, N, K, relu,
                                                           kAccChunk, whatif_value(OPT_WHATIF_LINEAR));
    note_launch();
    return cudaGetLastError();
}

// tile width: 128 columns, or 96 when that wastes fewer (N = 96, 192, 288 ...)
bool narrow_tile(int N) { return (N + 95) / 96 * 96 - N < (N + 127) / 128 * 128 - N; }

}  // namespace

// split[0 .. N*K) = tf32(w), split[N*K .. 2*N*K) = tf32(w - tf32(w)): what launch_linear_tf32x3 does per call when
// it is given the weight; done once by callers whose weight does not change between calls (inference)
cudaError_t launch_split_weight(const float *w, float *split, int N, int K, cudaStream_t stream, bool *handled) {
    *handled = false;
    if (N <= 0 || K <= 0 || ((long long)N * K) % 4 != 0 ||
        (reinterpret_cast<uintptr_t>(w) | reinterpret_cast<uintptr_t>(split)) % 16 != 0)
        return cudaSuccess;
    *handled = true;
    const long long n4 = (long long)N * K / 4;
    split_weight_kernel<<<(unsigned)((n4 + 255) / 256 < 592 ? (n4 + 255) / 256 : 592), 256, 0, stream>>>(
        reinterpret_cast<const float4 *>(w), reinterpret_cast<float4 *>(split),
        reinterpret_cast<float4 *>(split + (size_t)N * K), n4);
    note_launch();
    return cudaGetLastError();
}

// y[M, N] = x[M, K] * w[N, K]^T + bias[N]; K % 32 == 0, 16-byte aligned rows; workspace: 2*N*K floats.
// deterministic: every output tile is reduced by one CTA, split-K chunks in chunk order (bit-identical to the
// default outside split-K shapes)
cudaError_t launch_linear_tf32x3(const float *x, const float *w, const float *bias, float *y, int M, int N, int K,
                                 int relu, float *workspace, cudaStream_t stream, bool *handled, bool deterministic) {
    *handled = true;
    if (M <= 0 || N <= 0 || K <= 0 || K % kBK != 0 || N % 4 != 0 ||
        (reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(w) | reinterpret_cast<uintptr_t>(workspace) |
         reinterpret_cast<uintptr_t>(y)) % 16 != 0 ||
        ((long long)K * 4) % 16 != 0 || (w == nullptr && workspace == nullptr)) {
        *handled = false;
        return cudaSuccess;
    }
    if (w == nullptr) {             // pre-split weight in the workspace: the A-in-tensor-memory kernel only
        if (narrow_tile(N)) return launch_linear_atmem<96>(x, nullptr, bias, y, M, N, K, relu, workspace, stream);
        return launch_linear_atmem<128>(x, nullptr, bias, y, M, N, K, relu, workspace, stream);
    }
    const bool narrow = narrow_tile(N);
    const int variant = option_value(OPT_LINEAR_VARIANT);
    if (workspace == nullptr) {
        // one-shot weight: split inside the kernel; long reductions (the use case) -> four accumulators
        if (narrow) return launch_linear<96, 3, 1, 4, true>(x, w, bias, y, M, N, K, relu, workspace, stream, deterministic);
        return launch_linear<128, 3, 1, 4, true>(x, w, bias, y, M, N, K, relu, workspace, stream, deterministic);
    }
    // default: A operand in tensor memory (fastest; {main, small} accumulators, drained into registers every
    // 256 of the reduction so that the truncating accumulation never sees more than 64 MMAs per accumulator)
    if (variant == 4 || variant == 0) {
        if (narrow) return launch_linear_atmem<96>(x, w, bias, y, M, N, K, relu, workspace, stream);
        return launch_linear_atmem<128>(x, w, bias, y, M, N, K, relu, workspace, stream);
    }
    // both operands in shared memory, the products spread over four accumulators (one set: the epilogue is
    // not overlapped) -- the long-reduction kernel before the chunked accumulation above
    if (variant == 2) {
        if (narrow) return launch_linear<96, 3, 1, 4, false>(x, w, bias, y, M, N, K, relu, workspace, stream, deterministic);
        return launch_linear<128, 3, 1, 4, false>(x, w, bias, y, M, N, K, relu, workspace, stream, deterministic);
    }
    if (narrow) return launch_linear<96, 3, 2, 2, false>(x, w, bias, y, M, N, K, relu, workspace, stream, deterministic);
    return launch_linear<128, 3, 2, 2, false>(x, w, bias, y, M, N, K, relu, workspace, stream, deterministic);
}

}  // namespace msda

#ifdef MSDA_PROFILE_KNOBS
// profiling build only: read (and clear) the pipeline cycle counters
extern "C" int msda_b200_debug_linear_counters(unsigned long long *out16) {
    cudaError_t e = cudaMemcpyFromSymbol(out16, g_lin_dbg, sizeof(g_lin_dbg));
    if (e != cudaSuccess) return (int)e;
    unsigned long long zero[16] = {};
    return (int)cudaMemcpyToSymbol(g_lin_dbg, zero, sizeof(zero));
}
#endif
