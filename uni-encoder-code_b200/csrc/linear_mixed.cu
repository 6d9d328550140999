// linear_mixed.cu -- the encoder's nn.Linear layers under torch.autocast: bf16 / fp16 GEMMs on the sm_100a tensor
// cores (tcgen05.mma.kind::f16, fp32 accumulation in tensor memory).
//
//   linear_mixed_kernel        y16[M, N] = round16(relu?(x16 * w16^T + bias)), bias fp32 (may be NULL) added to the
//                              fp32 accumulator, one round-to-nearest-even at the end (fp16 overflow gives +-inf).
//                              Also the input gradient: grad_x16 = grad_y16 * w16 with the transposed weight.
//   linear_mixed_wgrad_kernel  fp32 partial grad_w = grad_y16^T * x16 and partial column sums of grad_y16 of one
//                              chunk of rows; wgrad_reduce_kernel adds the chunks in chunk order (deterministic by
//                              construction: no floating-point atomics anywhere).
//
// Forward structure (persistent: one CTA per SM walks 128 x BN output tiles, BN <= 256; 10 warps):
//   warp 0     one thread: TMA loads of the X tile (128 x 64) and the W tile (BN x 64) of each k-block into a
//              4-deep ring (128-byte swizzle: a tile row is one swizzle span);
//   warp 1     one elected thread: four tcgen05.mma of depth 16 per k-block into one of two accumulators in TMEM,
//              tcgen05.commit to release the stage, and the accumulator when the tile is complete;
//   warps 2-9  epilogue, two warps per TMEM lane quarter on alternate 32-column blocks: tcgen05.ld (lane = row),
//              bias, ReLU, rounding, then through shared memory into 64-byte row segments so that one store
//              instruction writes whole segments of 8 rows.  With two accumulators the epilogue of tile i overlaps
//              the MMAs of tile i+1.
// These GEMMs are bound by HBM at the encoder's shapes: the CTAs that compute the N tiles of one row block run
// side by side (tile index = row block * n_tiles + n tile), so the X rows come from HBM once and from L2 after.
//
// Weight gradient: the reduction runs over the rows, and 16-bit tcgen05 operands may be MN-major in shared memory,
// so TMA loads the row-major grad_y and x tiles as they are (64 rows x 64 columns per box) and the MMA reads them
// MN-major.  The bias sums come from a second MMA of the same grad_y tile against a constant tile of ones.
#include "tc_common.cuh"

namespace msda {

using namespace tc;

namespace {

template <typename T> struct Bits16;
template <> struct Bits16<__nv_bfloat16> {
    static constexpr bool kBf16 = true;
    static constexpr uint16_t kOne = 0x3f80;
    static __device__ __forceinline__ uint32_t pack(float a, float b) {
        const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
        return *reinterpret_cast<const uint32_t *>(&h);
    }
};
template <> struct Bits16<__half> {
    static constexpr bool kBf16 = false;
    static constexpr uint16_t kOne = 0x3c00;
    static __device__ __forceinline__ uint32_t pack(float a, float b) {
        const __half2 h = __floats2half2_rn(a, b);
        return *reinterpret_cast<const uint32_t *>(&h);
    }
};

// ---------------------------------------------------------------------------------------------------------------
// forward / input gradient
// ---------------------------------------------------------------------------------------------------------------
constexpr int kFwdStages = 4;
constexpr int kFwdMaxBN = 256;                 // also the TMEM column offset of the second accumulator
constexpr int kFwdEpiWarps = 8;
constexpr int kFwdThreads = 64 + 32 * kFwdEpiWarps;
constexpr int kEpiRow = 80;                    // bytes per staged row: 32 columns (64 bytes) + 16 (no bank conflicts)

struct FwdCfg {
    static constexpr int kXBytes = kBM * kBK16 * 2;
    static constexpr int kWBytes = kFwdMaxBN * kBK16 * 2;
    static constexpr int kStageBytes = kXBytes + kWBytes;
    static constexpr int kRingBytes = kFwdStages * kStageBytes;
    static constexpr int kEpiBytes = kFwdEpiWarps * 32 * kEpiRow;
    static constexpr int kSmem = kRingBytes + kEpiBytes + 1024 /* alignment slack */ + 256 /* barriers */;
};

template <typename T>
__global__ void __launch_bounds__(kFwdThreads, 1)
linear_mixed_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_w,
                    const float *__restrict__ bias, T *__restrict__ y, int M, int N, int K, int BN, int relu) {
    constexpr int STAGES = kFwdStages;
    extern __shared__ uint8_t smem_dyn[];
    const uint32_t base = (smem_u32(smem_dyn) + 1023u) & ~1023u;
    uint8_t *base_ptr = smem_dyn + (base - smem_u32(smem_dyn));
    const uint32_t bars = base + FwdCfg::kRingBytes + FwdCfg::kEpiBytes;
    // ring: full[s] (TMA landed), empty[s] (MMAs done); accumulators: acc_full[b] (tile complete), acc_empty[b]
    auto full = [&](int s) { return bars + 8u * s; };
    auto empty = [&](int s) { return bars + 8u * (STAGES + s); };
    auto acc_full = [&](int b) { return bars + 8u * (2 * STAGES + b); };
    auto acc_empty = [&](int b) { return bars + 8u * (2 * STAGES + 2 + b); };
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(base_ptr + FwdCfg::kRingBytes + FwdCfg::kEpiBytes +
                                                       8 * (2 * STAGES + 4));

    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    const int kblocks = (K + kBK16 - 1) / kBK16;
    const int n_tiles = (N + BN - 1) / BN;
    const long long tiles = (long long)((M + kBM - 1) / kBM) * n_tiles;

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(full(s), 1);
            mbar_init(empty(s), 1);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(acc_full(b), 1);
            mbar_init(acc_empty(b), kFwdEpiWarps);
        }
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
        if (lane == 0) {
            const uint32_t tx = FwdCfg::kXBytes + (uint32_t)BN * kBK16 * 2;   // zero-filled parts count as well
            uint32_t g = 0;
            for (long long t = blockIdx.x; t < tiles; t += gridDim.x) {
                const int m0 = (int)(t / n_tiles) * kBM, n0 = (int)(t % n_tiles) * BN;
                for (int kb = 0; kb < kblocks; ++kb, ++g) {
                    const int s = g % STAGES;
                    mbar_wait(empty(s), ((g / STAGES) & 1) ^ 1);
                    const uint32_t st = base + s * FwdCfg::kStageBytes;
                    mbar_arrive_expect_tx(full(s), tx);
                    tma_load_2d(st, &map_x, full(s), kb * kBK16, m0);
                    tma_load_2d(st + FwdCfg::kXBytes, &map_w, full(s), kb * kBK16, n0);
                }
            }
        }
    } else if (warp == 1) {
        const uint32_t idesc = umma_idesc_f16(kBM, BN, Bits16<T>::kBf16, false, false);
        const bool leader = elect_one();
        uint32_t g = 0, it = 0;
        for (long long t = blockIdx.x; t < tiles; t += gridDim.x, ++it) {
            const uint32_t buf = it & 1;
            mbar_wait(acc_empty(buf), ((it >> 1) & 1) ^ 1);                 // the epilogue has drained it
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t acc = tmem_base + buf * kFwdMaxBN;
            for (int kb = 0; kb < kblocks; ++kb, ++g) {
                const int s = g % STAGES;
                mbar_wait(full(s), (g / STAGES) & 1);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t xa = base + s * FwdCfg::kStageBytes, wa = xa + FwdCfg::kXBytes;
                if (leader) {
#pragma unroll
                    for (int k = 0; k < kBK16 / kUmmaK16; ++k)            // + 32 bytes inside the swizzle span
                        umma_f16(acc, umma_desc(xa + k * 32), umma_desc(wa + k * 32), idesc, (kb | k) != 0);
                    umma_commit(empty(s));
                }
                __syncwarp();
            }
            if (leader) umma_commit(acc_full(buf));
            __syncwarp();
        }
    } else {
        const int ew = warp - 2, q = warp & 3, part = ew >> 2;
        uint8_t *stage = base_ptr + FwdCfg::kRingBytes + ew * 32 * kEpiRow;
        const int sub = lane >> 2, ch = lane & 3;                          // store loop: row in a group of 8, chunk
        uint32_t it = 0;
        for (long long t = blockIdx.x; t < tiles; t += gridDim.x, ++it) {
            const int m0 = (int)(t / n_tiles) * kBM, n0 = (int)(t % n_tiles) * BN;
            const uint32_t buf = it & 1;
            mbar_wait(acc_full(buf), (it >> 1) & 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t acc = tmem_base + buf * kFwdMaxBN + ((uint32_t)(q * 32) << 16);
            for (int c = part; c < BN / 32; c += 2) {
                uint32_t v[32];
                tmem_ld32(acc + (uint32_t)(c * 32), v);
                const int col0 = n0 + c * 32;
                const float bl = (bias != nullptr && col0 + lane < N) ? bias[col0 + lane] : 0.f;
                uint32_t p[16];
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    float a = __uint_as_float(v[2 * j]) + __shfl_sync(0xffffffffu, bl, 2 * j);
                    float b = __uint_as_float(v[2 * j + 1]) + __shfl_sync(0xffffffffu, bl, 2 * j + 1);
                    if (relu) {                                            // NaN stays NaN, as in F.relu
                        a = a < 0.f ? 0.f : a;
                        b = b < 0.f ? 0.f : b;
                    }
                    p[j] = Bits16<T>::pack(a, b);
                }
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    *reinterpret_cast<uint4 *>(stage + lane * kEpiRow + j * 16) =
                        make_uint4(p[4 * j], p[4 * j + 1], p[4 * j + 2], p[4 * j + 3]);
                __syncwarp();
                const int col = col0 + ch * 8;
#pragma unroll
                for (int r8 = 0; r8 < 4; ++r8) {
                    const int r = r8 * 8 + sub, row = m0 + q * 32 + r;
                    const uint4 o = *reinterpret_cast<const uint4 *>(stage + r * kEpiRow + ch * 16);
                    if (row < M && col < N) *reinterpret_cast<uint4 *>(y + (long long)row * N + col) = o;
                }
                __syncwarp();
            }
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(acc_empty(buf));
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
}

// ---------------------------------------------------------------------------------------------------------------
// weight + bias gradient
// ---------------------------------------------------------------------------------------------------------------
constexpr int kWgStages = 4;
constexpr int kWgMaxBN = 256;                  // in_features per tile
constexpr int kWgEpiWarps = 4;
constexpr int kWgThreads = 64 + 32 * kWgEpiWarps;
constexpr int kBox = 64 * kBK16 * 2;           // one TMA box: 64 rows x 64 columns (8 KB)
constexpr int kBiasCol = kWgMaxBN;             // TMEM column of the bias sums
// work items a call is split into: one wave of 148 CTAs (a B200's SMs).  A constant rather than the device's SM
// count, so that the chunking -- and with it every bit of the result -- depends on the shapes alone.
constexpr int kWgItems = 148;

struct WgCfg {
    static constexpr int kABytes = 2 * kBox;                          // grad_y: 64 rows x 128 out
    static constexpr int kBBytes = (kWgMaxBN / 64) * kBox;            // x: 64 rows x 256 in
    static constexpr int kStageBytes = kABytes + kBBytes;
    static constexpr int kRingBytes = kWgStages * kStageBytes;
    static constexpr int kOnesBytes = 16 * 128;                       // B operand of the bias MMA: 16 x 64 ones
    static constexpr int kSmem = kRingBytes + kOnesBytes + 1024 + 256;
};

struct WgPlan {
    int bn, n_tiles, m_tiles, kblocks, kb_per_chunk, chunks;
};

WgPlan wgrad_plan(long long rows, int out_f, int in_f) {
    WgPlan p;
    p.n_tiles = (in_f + kWgMaxBN - 1) / kWgMaxBN;
    p.bn = ((in_f + p.n_tiles - 1) / p.n_tiles + 63) / 64 * 64;
    p.n_tiles = (in_f + p.bn - 1) / p.bn;
    p.m_tiles = (out_f + kBM - 1) / kBM;
    p.kblocks = (int)((rows + kBK16 - 1) / kBK16);
    const int tiles = p.n_tiles * p.m_tiles;
    int chunks = kWgItems / tiles;
    if (chunks < 1) chunks = 1;
    if (chunks > p.kblocks) chunks = p.kblocks;
    p.kb_per_chunk = (p.kblocks + chunks - 1) / chunks;
    p.chunks = (p.kblocks + p.kb_per_chunk - 1) / p.kb_per_chunk;
    return p;
}

// grid: n_tiles * m_tiles * chunks CTAs, tile fastest (the CTAs of one chunk read the same rows side by side);
// partial[chunk][out_f][in_f], partial_b[chunk][out_f]
template <typename T>
__global__ void __launch_bounds__(kWgThreads, 1)
linear_mixed_wgrad_kernel(const __grid_constant__ CUtensorMap map_g, const __grid_constant__ CUtensorMap map_x,
                          float *__restrict__ partial, float *__restrict__ partial_b, int out_f, int in_f, int BN,
                          int n_tiles, int m_tiles, int kblocks, int kb_per_chunk) {
    constexpr int STAGES = kWgStages;
    extern __shared__ uint8_t smem_dyn[];
    const uint32_t base = (smem_u32(smem_dyn) + 1023u) & ~1023u;
    uint8_t *base_ptr = smem_dyn + (base - smem_u32(smem_dyn));
    const uint32_t ones = base + WgCfg::kRingBytes;
    const uint32_t bars = ones + WgCfg::kOnesBytes;
    auto full = [&](int s) { return bars + 8u * s; };
    auto empty = [&](int s) { return bars + 8u * (STAGES + s); };
    const uint32_t acc_full = bars + 8u * 2 * STAGES;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(base_ptr + WgCfg::kRingBytes + WgCfg::kOnesBytes +
                                                       8 * (2 * STAGES + 1));

    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    const int tiles = n_tiles * m_tiles;
    const int tile = (int)(blockIdx.x % (unsigned)tiles), chunk = (int)(blockIdx.x / (unsigned)tiles);
    const int m0 = (tile / n_tiles) * kBM, n0 = (tile % n_tiles) * BN;
    const int kb0 = chunk * kb_per_chunk, nkb = min(kb_per_chunk, kblocks - kb0);
    const bool with_bias = partial_b != nullptr && n0 == 0;

    {
        uint32_t *o = reinterpret_cast<uint32_t *>(base_ptr + WgCfg::kRingBytes);
        const uint32_t one2 = (uint32_t)Bits16<T>::kOne * 0x10001u;
        for (int i = threadIdx.x; i < WgCfg::kOnesBytes / 4; i += blockDim.x) o[i] = one2;
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");       // generic writes -> tensor core reads
    }
    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(full(s), 1);
            mbar_init(empty(s), 1);
        }
        mbar_init(acc_full, 1);
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
        if (lane == 0) {
            // boxes that start past the matrix are not loaded: their rows / columns of the result are not stored
            const int a_boxes = min(2, (out_f - m0 + 63) / 64), b_boxes = min(BN / 64, (in_f - n0 + 63) / 64);
            const uint32_t tx = (uint32_t)(a_boxes + b_boxes) * kBox;
            for (int kb = 0; kb < nkb; ++kb) {
                const int s = kb % STAGES, r0 = (kb0 + kb) * kBK16;
                mbar_wait(empty(s), ((kb / STAGES) & 1) ^ 1);
                const uint32_t st = base + s * WgCfg::kStageBytes;
                mbar_arrive_expect_tx(full(s), tx);
                for (int h = 0; h < a_boxes; ++h) tma_load_2d(st + h * kBox, &map_g, full(s), m0 + h * 64, r0);
                for (int h = 0; h < b_boxes; ++h)
                    tma_load_2d(st + WgCfg::kABytes + h * kBox, &map_x, full(s), n0 + h * 64, r0);
            }
        }
    } else if (warp == 1) {
        const uint32_t idesc = umma_idesc_f16(kBM, BN, Bits16<T>::kBf16, true, true);
        const uint32_t idesc_b = umma_idesc_f16(kBM, 16, Bits16<T>::kBf16, true, false);
        const bool leader = elect_one();
        for (int kb = 0; kb < nkb; ++kb) {
            const int s = kb % STAGES;
            mbar_wait(full(s), (kb / STAGES) & 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t sa = base + s * WgCfg::kStageBytes, sb = sa + WgCfg::kABytes;
            if (leader) {
#pragma unroll
                for (int k = 0; k < kBK16 / kUmmaK16; ++k) {               // 16 rows = two 1024-byte atoms per step
                    const uint64_t da = umma_desc_mn(sa + k * 2048, kBox);
                    umma_f16(tmem_base, da, umma_desc_mn(sb + k * 2048, kBox), idesc, (kb | k) != 0);
                    if (with_bias) umma_f16(tmem_base + kBiasCol, da, umma_desc(ones + k * 32), idesc_b, (kb | k) != 0);
                }
                umma_commit(empty(s));
            }
            __syncwarp();
        }
        if (leader) umma_commit(acc_full);
        __syncwarp();
    } else {
        const int q = warp & 3, row = m0 + q * 32 + lane;
        const uint32_t acc = tmem_base + ((uint32_t)(q * 32) << 16);
        mbar_wait(acc_full, 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        float *dst = partial + ((long long)chunk * out_f + row) * in_f;
        for (int c = 0; c < BN / 32; ++c) {
            uint32_t v[32];
            tmem_ld32(acc + (uint32_t)(c * 32), v);
            if (row < out_f) {
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int col = n0 + c * 32 + 4 * j;
                    if (col < in_f)
                        *reinterpret_cast<float4 *>(dst + col) = make_float4(
                            __uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]), __uint_as_float(v[4 * j + 2]),
                            __uint_as_float(v[4 * j + 3]));
                }
            }
        }
        if (with_bias) {
            uint32_t v[32];
            tmem_ld32(acc + (uint32_t)kBiasCol, v);
            if (row < out_f) partial_b[(long long)chunk * out_f + row] = __uint_as_float(v[0]);
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
}

// grad_w = sum of the chunks' partial tiles, grad_b = sum of their bias partials, each added in chunk order
__global__ void linear_mixed_wgrad_reduce_kernel(const float4 *__restrict__ partial, float4 *__restrict__ grad_w,
                                                 long long n4, const float *__restrict__ partial_b,
                                                 float *__restrict__ grad_b, int out_f, int chunks) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
        float4 s = partial[i];
        for (int c = 1; c < chunks; ++c) {
            const float4 v = partial[(long long)c * n4 + i];
            s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
        }
        grad_w[i] = s;
    }
    if (grad_b != nullptr) {
        for (long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x; o < out_f; o += stride) {
            float s = partial_b[o];
            for (int c = 1; c < chunks; ++c) s += partial_b[(long long)c * out_f + o];
            grad_b[o] = s;
        }
    }
}

template <typename K>
cudaError_t set_smem_once(K kern, int bytes, std::atomic<bool> (&attr_set)[kMaxDevices]) {
    cudaError_t e = cudaSuccess;
    const int dev = device_slot(&e);
    if (dev < 0) return e;
    if (!attr_set[dev].load(std::memory_order_acquire)) {
        e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
        if (e != cudaSuccess) return e;
        attr_set[dev].store(true, std::memory_order_release);
    }
    return cudaSuccess;
}

bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

}  // namespace

// y[M, N] = round16(relu?(x[M, K] * w[N, K]^T + bias)); K % 8 == 0, N % 8 == 0, 16-byte aligned x, w, y
template <typename T>
cudaError_t launch_linear_mixed(const T *x, const T *w, const float *bias, T *y, int M, int N, int K, int relu,
                                cudaStream_t stream, bool *handled) {
    *handled = false;
    if (K % 8 != 0 || N % 8 != 0 || !aligned16(x) || !aligned16(w) || !aligned16(y)) return cudaSuccess;
    *handled = true;
    auto kern = linear_mixed_kernel<T>;
    static std::atomic<bool> attr_set[kMaxDevices];
    cudaError_t e = set_smem_once(kern, FwdCfg::kSmem, attr_set);
    if (e != cudaSuccess) return e;
    // the fewest tiles of at most 256 columns, as equal as 32-column blocks make them (288 -> 2 x 160)
    const int n_tiles = (N + kFwdMaxBN - 1) / kFwdMaxBN;
    const int bn = ((N + n_tiles - 1) / n_tiles + 31) / 32 * 32;
    CUtensorMap mx, mw;
    if (!make_map16(&mx, x, M, K, kBM, Bits16<T>::kBf16) || !make_map16(&mw, w, N, K, bn, Bits16<T>::kBf16))
        return cudaErrorInvalidValue;
    const long long tiles = (long long)((M + kBM - 1) / kBM) * ((N + bn - 1) / bn);
    const long long grid = tiles < sm_count() ? tiles : sm_count();
    kern<<<(unsigned)grid, kFwdThreads, FwdCfg::kSmem, stream>>>(mx, mw, bias, y, M, N, K, bn, relu);
    note_launch();
    return cudaGetLastError();
}

long long linear_mixed_wgrad_workspace_floats(long long rows, int out_f, int in_f) {
    const WgPlan p = wgrad_plan(rows, out_f, in_f);
    return (long long)p.chunks * ((long long)out_f * in_f + out_f);
}

// grad_w[out_f, in_f] = grad_y[rows, out_f]^T * x[rows, in_f], grad_b[out_f] = column sums of grad_y (may be NULL);
// out_f % 8 == 0, in_f % 8 == 0, 16-byte aligned operands and workspace
template <typename T>
cudaError_t launch_linear_mixed_wgrad(const T *grad_y, const T *x, float *grad_w, float *grad_b, long long rows,
                                      int out_f, int in_f, float *workspace, cudaStream_t stream, bool *handled) {
    *handled = false;
    if (out_f % 8 != 0 || in_f % 8 != 0 || !aligned16(grad_y) || !aligned16(x) || !aligned16(grad_w) ||
        !aligned16(workspace))
        return cudaSuccess;
    *handled = true;
    auto kern = linear_mixed_wgrad_kernel<T>;
    static std::atomic<bool> attr_set[kMaxDevices];
    cudaError_t e = set_smem_once(kern, WgCfg::kSmem, attr_set);
    if (e != cudaSuccess) return e;
    const WgPlan p = wgrad_plan(rows, out_f, in_f);
    CUtensorMap mg, mx;
    if (!make_map16(&mg, grad_y, rows, out_f, 64, Bits16<T>::kBf16) ||
        !make_map16(&mx, x, rows, in_f, 64, Bits16<T>::kBf16))
        return cudaErrorInvalidValue;
    float *partial_b = workspace + (long long)p.chunks * out_f * in_f;
    const unsigned grid = (unsigned)(p.n_tiles * p.m_tiles * p.chunks);
    kern<<<grid, kWgThreads, WgCfg::kSmem, stream>>>(mg, mx, workspace, grad_b != nullptr ? partial_b : nullptr, out_f,
                                                     in_f, p.bn, p.n_tiles, p.m_tiles, p.kblocks, p.kb_per_chunk);
    note_launch();
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    const long long n4 = (long long)out_f * in_f / 4;
    const long long blocks = (n4 + 255) / 256;
    linear_mixed_wgrad_reduce_kernel<<<(unsigned)(blocks < 4 * sm_count() ? blocks : 4 * sm_count()), 256, 0, stream>>>(
        reinterpret_cast<const float4 *>(workspace), reinterpret_cast<float4 *>(grad_w), n4, partial_b, grad_b, out_f,
        p.chunks);
    note_launch();
    return cudaGetLastError();
}

template cudaError_t launch_linear_mixed<__nv_bfloat16>(const __nv_bfloat16 *, const __nv_bfloat16 *, const float *,
                                                        __nv_bfloat16 *, int, int, int, int, cudaStream_t, bool *);
template cudaError_t launch_linear_mixed<__half>(const __half *, const __half *, const float *, __half *, int, int,
                                                 int, int, cudaStream_t, bool *);
template cudaError_t launch_linear_mixed_wgrad<__nv_bfloat16>(const __nv_bfloat16 *, const __nv_bfloat16 *, float *,
                                                              float *, long long, int, int, float *, cudaStream_t,
                                                              bool *);
template cudaError_t launch_linear_mixed_wgrad<__half>(const __half *, const __half *, float *, float *, long long, int,
                                                       int, float *, cudaStream_t, bool *);

}  // namespace msda
