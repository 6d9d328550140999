// linear_wgrad.cu -- weight (and bias) gradient of an fp32 nn.Linear on the sm_100a tensor cores:
//     grad_W[out, in] = grad_y[rows, out]^T * x[rows, in],      grad_b[out] = column sums of grad_y
// with the same error-compensated 3xTF32 scheme as linear_tf32x3.cu (see there), WITHOUT transposing the
// operands in global memory.
//
// The reduction runs over the rows, which are the slow dimension of both row-major operands, so neither is
// "K-major".  Per k-block of 32 rows TMA loads the plain tiles grad_y[32, 128] and x[32, BN] (no swizzle);
// the four operand warps then
//   * read column n of the grad_y tile (lane = n: conflict-free 128-byte reads) and tcgen05.st its 32 values
//     -- hi as they are, lo = tf32(v - trunc19(v)) -- into the A ring in tensor memory (lane = row of A = n,
//     32 columns = the 32 rows of the k-block), adding them up on the way for grad_b;
//   * read column k of the x tile the same way and write it as one 128-byte row of the K-major, 128-byte
//     swizzled B tiles B_hi / B_lo in shared memory (what a K-major TMA load would have produced);
// and the MMA thread issues x-like products from there: A_hi * [B_hi; B_lo]^T -> {main, small}, A_lo * B_hi^T ->
// small.  An output tile (128 x BN of grad_W) is computed by several work items, each over a chunk of the rows
// (split-K), and added into the zero-filled output with red.global.add -- or, in the deterministic entry, stored
// as the chunk's partial tile in a workspace whose chunks a second launch adds up in chunk order.
#include "tc_common.cuh"

namespace msda {

using namespace tc;

namespace {

constexpr int kOpWarps = 4;       // warps 2-5: operand preparation (one per TMEM lane quarter)
constexpr int kEpiWarps = 8;      // warps 6-13
constexpr int kThreads = 64 + 32 * (kOpWarps + kEpiWarps);
constexpr int kStages = 3;

template <int BN>
struct WgCfg {
    static constexpr int kYBytes = kBK * kBM * 4;                  // grad_y tile [32 rows][128 outs]
    static constexpr int kXBytes = kBK * BN * 4;                   // x tile      [32 rows][BN ins]
    static constexpr int kBBytes = BN * kBK * 4;                   // B_hi or B_lo: [BN ins][32 rows], K-major
    static constexpr int kStageBytes = kYBytes + kXBytes + 2 * kBBytes;
    static constexpr int kRingBytes = kStages * kStageBytes;
    static constexpr int kEpiBytes = kEpiWarps * 32 * 33 * 4;
    static constexpr int kSmem = kRingBytes + kEpiBytes + 1024 + 256;
    static constexpr int kACol = 2 * BN;                           // TMEM: {main, small}, then the A ring
    static_assert(2 * BN + kStages * 64 <= 512 && kStageBytes % 1024 == 0 && BN == 128, "tile shape");
};

template <int BN>
__global__ void __launch_bounds__(kThreads, 1)
linear_wgrad_kernel(const __grid_constant__ CUtensorMap map_gy, const __grid_constant__ CUtensorMap map_x,
                    float *__restrict__ grad_w, float *__restrict__ grad_b, long long rows, int out_f, int in_f,
                    int chunks, int kb_per_chunk, float *__restrict__ partials) {
    using Cfg = WgCfg<BN>;
    extern __shared__ uint8_t smem_dyn[];
    const uint32_t base = (smem_u32(smem_dyn) + 1023u) & ~1023u;
    uint8_t *base_ptr = smem_dyn + (base - smem_u32(smem_dyn));
    const uint32_t bars = base + Cfg::kRingBytes + Cfg::kEpiBytes;
    auto full = [&](int s) { return bars + 8u * s; };
    auto ready = [&](int s) { return bars + 8u * (kStages + s); };
    auto empty = [&](int s) { return bars + 8u * (2 * kStages + s); };
    const uint32_t acc_full = bars + 8u * 3 * kStages, acc_empty = acc_full + 8u;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(base_ptr + Cfg::kRingBytes + Cfg::kEpiBytes + 8 * (3 * kStages + 2));

    // the warp index through a shuffle: provably warp-uniform, so the role loops stay in uniform registers
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    const int kblocks_all = (int)((rows + kBK - 1) / kBK);
    const int n_tiles = (out_f + kBM - 1) / kBM, k_tiles = (in_f + BN - 1) / BN;
    // work items: (row chunk, output tile), output tile fastest -- the items that read the same rows of grad_y
    // and x run at the same time on neighbouring SMs, so each row is fetched from HBM once (chunk fastest
    // measured 2x the DRAM reads: every operand came in once per output-tile row / column)
    const long long items = (long long)n_tiles * k_tiles * chunks;
    auto decode = [&](long long t, int &n0, int &k0, int &kb0, int &nkb) {
        const int out_tiles = n_tiles * k_tiles;
        const int chunk = (int)(t / out_tiles);
        const long long o = t % out_tiles;
        n0 = (int)(o / k_tiles) * kBM;
        k0 = (int)(o % k_tiles) * BN;
        kb0 = chunk * kb_per_chunk;
        nkb = min(kb_per_chunk, kblocks_all - kb0);
    };

    if (threadIdx.x == 0) {
        for (int s = 0; s < kStages; ++s) {
            mbar_init(full(s), 1);
            mbar_init(ready(s), 32 * kOpWarps);
            mbar_init(empty(s), 1);
        }
        mbar_init(acc_full, 1);
        mbar_init(acc_empty, 32 * kEpiWarps);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     ::"r"(smem_u32(tmem_slot)), "r"(512) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);

    if (warp == 0) {
        // ---- TMA producer: plain tiles of grad_y and x, 32 rows each ----
        if (lane == 0) {
            uint32_t g = 0;
            for (long long t = blockIdx.x; t < items; t += gridDim.x) {
                int n0, k0, kb0, nkb;
                decode(t, n0, k0, kb0, nkb);
                for (int kb = 0; kb < nkb; ++kb, ++g) {
                    const int s = g % kStages;
                    mbar_wait(empty(s), ((g / kStages) & 1) ^ 1);
                    const uint32_t st = base + s * Cfg::kStageBytes;
                    mbar_arrive_expect_tx(full(s), Cfg::kYBytes + Cfg::kXBytes);
                    tma_load_2d(st, &map_gy, full(s), n0, (kb0 + kb) * kBK);
                    tma_load_2d(st + Cfg::kYBytes, &map_x, full(s), k0, (kb0 + kb) * kBK);
                }
            }
        }
    } else if (warp == 1) {
        // ---- MMA issuer: the whole warp walks the loop (warp-uniform control flow keeps the descriptors in uniform
        //      registers: the 8 tcgen05.mma of a k-block issue back to back -- an MMA is accepted only when the previous
        //      one is nearly done, so instructions between two issues are tensor-core idle time); one elected lane issues
        constexpr uint32_t idesc = umma_idesc(kBM, BN), idesc2 = umma_idesc(kBM, 2 * BN);
        const bool leader = elect_one();
        uint32_t g = 0, it = 0;
        for (long long t = blockIdx.x; t < items; t += gridDim.x, ++it) {
            int n0, k0, kb0, nkb;
            decode(t, n0, k0, kb0, nkb);
            mbar_wait(acc_empty, (it & 1) ^ 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            for (int kb = 0; kb < nkb; ++kb, ++g) {
                const int s = g % kStages;
                mbar_wait(ready(s), (g / kStages) & 1);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint64_t db0 = umma_desc(base + s * Cfg::kStageBytes + Cfg::kYBytes + Cfg::kXBytes);
                const uint32_t a_hi = tmem_base + Cfg::kACol + s * 64, a_lo = a_hi + 32;
                if (leader) {
#pragma unroll
                    for (int k = 0; k < kBK / kUmmaK; ++k) {
                        const uint64_t db = db0 + (uint64_t)((k * kUmmaK * 4) >> 4);   // + 32 bytes per k-step (address field)
                        umma_tf32_ts(tmem_base, a_hi + k * kUmmaK, db, idesc2, (kb | k) != 0);
                        umma_tf32_ts(tmem_base + BN, a_lo + k * kUmmaK, db, idesc, 1);
                    }
                    umma_commit(empty(s));
                }
            }
            if (leader) umma_commit(acc_full);
        }
    } else if (warp < 2 + kOpWarps) {
        // ---- operand warps ----
        const int q = warp & 3, col = q * 32 + lane;                  // A row / B row handled by this thread
        uint32_t g = 0;
        for (long long t = blockIdx.x; t < items; t += gridDim.x) {
            int n0, k0, kb0, nkb;
            decode(t, n0, k0, kb0, nkb);
            float bsum = 0.f;
            for (int kb = 0; kb < nkb; ++kb, ++g) {
                const int s = g % kStages;
                mbar_wait(full(s), (g / kStages) & 1);
                const float *ty = reinterpret_cast<const float *>(base_ptr + s * Cfg::kStageBytes);
                const float *tx = reinterpret_cast<const float *>(base_ptr + s * Cfg::kStageBytes + Cfg::kYBytes);
                uint8_t *bhi = base_ptr + s * Cfg::kStageBytes + Cfg::kYBytes + Cfg::kXBytes + col * 128;
                uint32_t hi[32], lo[32];
                // A = grad_y^T: row `col` of A is column `col` of the tile
#pragma unroll
                for (int m = 0; m < 32; ++m) {
                    const float v = ty[m * kBM + col];
                    bsum += v;
                    hi[m] = __float_as_uint(v);
                    lo[m] = to_tf32(v - __uint_as_float(hi[m] & 0xffffe000u));
                }
                const uint32_t a_hi = tmem_base + ((uint32_t)(q * 32) << 16) + Cfg::kACol + s * 64;
                tmem_st32(a_hi, hi);
                tmem_st32(a_hi + 32, lo);
                // B = x^T: row `col` of B (K-major, 128 bytes, chunk j stored at j ^ (row % 8)) is column `col` of the tile
#pragma unroll
                for (int m = 0; m < 32; ++m) {
                    const float v = tx[m * BN + col];
                    hi[m] = __float_as_uint(v);
                    lo[m] = to_tf32(v - __uint_as_float(hi[m] & 0xffffe000u));
                }
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int pos = (j ^ (col & 7)) << 4;
                    *reinterpret_cast<uint4 *>(bhi + pos) = make_uint4(hi[4 * j], hi[4 * j + 1], hi[4 * j + 2], hi[4 * j + 3]);
                    *reinterpret_cast<uint4 *>(bhi + Cfg::kBBytes + pos) = make_uint4(lo[4 * j], lo[4 * j + 1], lo[4 * j + 2], lo[4 * j + 3]);
                }
                asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                mbar_arrive(ready(s));
            }
            // bias gradient: every (out tile, chunk) contributes once (taken from the first in-tile)
            if (grad_b != nullptr && k0 == 0 && n0 + col < out_f) {
                if (partials != nullptr)
                    partials[(long long)chunks * out_f * in_f + (long long)(kb0 / kb_per_chunk) * out_f + n0 + col] = bsum;
                else
                    asm volatile("red.global.add.f32 [%0], %1;" ::"l"(grad_b + n0 + col), "f"(bsum) : "memory");
            }
        }
    } else {
        // ---- epilogue warps: accumulators -> registers (set handed back at once) -> transposes -> reductions ----
        const int q = warp & 3;
        float *tile = reinterpret_cast<float *>(base_ptr + Cfg::kRingBytes) + (warp - 2 - kOpWarps) * 32 * 33;
        uint32_t it = 0;
        for (long long t = blockIdx.x; t < items; t += gridDim.x, ++it) {
            int n0, k0, kb0, nkb;
            decode(t, n0, k0, kb0, nkb);
            const uint32_t acc = tmem_base + ((uint32_t)(q * 32) << 16);
            float *chunk_out = partials != nullptr ? partials + (long long)(kb0 / kb_per_chunk) * out_f * in_f : nullptr;
            mbar_wait(acc_full, it & 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            constexpr int kStep = kEpiWarps / 4, kMaxBlk = (BN / 32 + kStep - 1) / kStep;
            const int part = (warp - 2 - kOpWarps) >> 2;
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
                }
            }
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            mbar_arrive(acc_empty);
#pragma unroll
            for (int i = 0; i < kMaxBlk; ++i) {
                const int c = part + i * kStep;
                if (c >= BN / 32) continue;
                const int colk = k0 + c * 32;
#pragma unroll
                for (int j = 0; j < 32; ++j) tile[lane * 33 + j] = sum[i][j];
                __syncwarp();
#pragma unroll 8
                for (int r = 0; r < 32; ++r) {
                    const int n = n0 + q * 32 + r;
                    const float o = tile[r * 33 + lane];
                    if (n < out_f && colk + lane < in_f) {
                        if (chunk_out != nullptr) chunk_out[(long long)n * in_f + colk + lane] = o;
                        else asm volatile("red.global.add.f32 [%0], %1;" ::"l"(grad_w + (long long)n * in_f + colk + lane), "f"(o));
                    }
                }
                __syncwarp();
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
}

// deterministic entry: out[i] = sum of the chunks' partials in chunk order (grad_w, then grad_b)
__global__ void __launch_bounds__(256)
linear_wgrad_sum_kernel(const float *__restrict__ partials, float *__restrict__ grad_w, float *__restrict__ grad_b,
                        int chunks, long long nw, int nb) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nw + (grad_b != nullptr ? nb : 0);
         i += (long long)gridDim.x * blockDim.x) {
        const bool is_w = i < nw;
        const float *p = is_w ? partials + i : partials + (long long)chunks * nw + (i - nw);
        const long long stride = is_w ? nw : nb;
        float s = 0.f;
        for (int c = 0; c < chunks; ++c) s += p[c * stride];
        if (is_w) grad_w[i] = s;
        else grad_b[i - nw] = s;
    }
}

// rows per work item: the tensor core truncates when it adds into the fp32 accumulators, so the error
// grows with the number of MMAs per accumulator -- 16 k-blocks (512 rows, 64 MMAs) per item keep it at
// the level of an fp32 SIMT GEMM (73 k-blocks measured 5x that); more items than 2 per SM are welcome
int wgrad_kb_per_chunk(long long rows) {
    const int kblocks = (int)((rows + kBK - 1) / kBK);
    int kb_per_chunk = option_value(OPT_WGRAD_CHUNK) > 0 ? option_value(OPT_WGRAD_CHUNK) : 16;   // "wgrad_chunk" option
    if (kb_per_chunk < 1) kb_per_chunk = 1;
    if (kb_per_chunk > kblocks) kb_per_chunk = kblocks;
    return kb_per_chunk;
}

}  // namespace

// floats of the deterministic entry's workspace: one partial grad_w and grad_b per row chunk
long long linear_wgrad_partials(long long rows, int out_f, int in_f) {
    const long long kblocks = (rows + kBK - 1) / kBK, kbpc = wgrad_kb_per_chunk(rows);
    return (kblocks + kbpc - 1) / kbpc * ((long long)out_f * in_f + out_f);
}

// grad_w[out_f, in_f] = grad_y[rows, out_f]^T x[rows, in_f]; grad_b[out_f] (optional) = column sums of grad_y.
// Both outputs are overwritten: zero-filled and reduced into, or, with `partials` (linear_wgrad_partials floats),
// summed from the per-chunk partial tiles in chunk order.  out_f % 4 == 0, in_f % 4 == 0, 16-byte aligned operands.
cudaError_t launch_linear_wgrad(const float *grad_y, const float *x, float *grad_w, float *grad_b, long long rows,
                                int out_f, int in_f, cudaStream_t stream, bool *handled, float *partials) {
    *handled = true;
    if (rows <= 0 || out_f <= 0 || in_f <= 0 || out_f % 4 != 0 || in_f % 4 != 0 || rows > 0x7fffffffLL ||
        (reinterpret_cast<uintptr_t>(grad_y) | reinterpret_cast<uintptr_t>(x)) % 16 != 0) {
        *handled = false;
        return cudaSuccess;
    }
    constexpr int BN = 128;
    using Cfg = WgCfg<BN>;
    auto kern = linear_wgrad_kernel<BN>;
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
    CUtensorMap mgy, mx;
    if (!make_map_plain(&mgy, grad_y, rows, out_f, kBK, kBM) || !make_map_plain(&mx, x, rows, in_f, kBK, BN))
        return cudaErrorInvalidValue;
    if (partials == nullptr) {
        cudaError_t e = cudaMemsetAsync(grad_w, 0, (size_t)out_f * in_f * sizeof(float), stream);
        if (e == cudaSuccess && grad_b != nullptr) e = cudaMemsetAsync(grad_b, 0, (size_t)out_f * sizeof(float), stream);
        if (e != cudaSuccess) return e;
    }
    const int kblocks = (int)((rows + kBK - 1) / kBK);
    const long long out_tiles = (long long)((out_f + kBM - 1) / kBM) * ((in_f + BN - 1) / BN);
    const int kb_per_chunk = wgrad_kb_per_chunk(rows);
    const long long chunks = (kblocks + kb_per_chunk - 1) / kb_per_chunk;
    const long long items = out_tiles * chunks;
    const long long grid = items < sm_count() ? items : sm_count();
    kern<<<(unsigned)grid, kThreads, Cfg::kSmem, stream>>>(mgy, mx, grad_w, grad_b, rows, out_f, in_f, (int)chunks,
                                                           kb_per_chunk, partials);
    note_launch();
    if (partials == nullptr) return cudaGetLastError();
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    const long long nw = (long long)out_f * in_f, total = nw + (grad_b != nullptr ? out_f : 0);
    const long long blocks = (total + 255) / 256 < (long long)sm_count() * 8 ? (total + 255) / 256 : (long long)sm_count() * 8;
    linear_wgrad_sum_kernel<<<(unsigned)blocks, 256, 0, stream>>>(partials, grad_w, grad_b, (int)chunks, nw, out_f);
    note_launch();
    return cudaGetLastError();
}

}  // namespace msda
