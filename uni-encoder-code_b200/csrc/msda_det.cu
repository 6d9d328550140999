// msda_det.cu -- deterministic grad_value for the MSDA backward (torch.use_deterministic_algorithms).
//
// The default backward adds every (sampling point, corner) contribution into grad_value with
// floating-point reductions whose order depends on scheduling.  Here grad_value is a gather by
// destination whose order is fixed by a stable sort:
//   1. records   the backward kernel of the path (msda_bwd.cu plain / fused, msda_generic.cu) runs in its
//                RECORDS mode: grad_sampling_loc / grad_attn_weight exactly as in the default mode, and for
//                every corner a record {destination row, weight} in its fixed slot (DetRecords,
//                msda_common.cuh);
//   2. sort      cub::DeviceRadixSort::SortPairs of (destination row, slot) over the bit width of N*S*M.  The
//                sort is stable and the slots enter in ascending order, so each row's records come out in
//                slot order: query, head, level, point, corner -- the order of a sequential loop;
//   3. bounds    a boundary pass over the sorted keys writes the first record of every row (no atomics);
//   4. gather    one warp per grad_value row (lane = channel, channel blocks of 32 beyond D = 32) adds
//                w[slot] * grad_output[query row of slot] in bucket order and writes the row; rows without
//                records are written as zeros, so grad_value needs no zero-fill.
// The records of a corner outside its level carry the key N*S*M and sort behind every real row.
// Nothing here allocates or reads back to the host: the sort's temporary storage is part of the caller's
// workspace, so the whole sequence can be captured into a CUDA graph.
#include <cub/device/device_radix_sort.cuh>

#include "msda_common.cuh"

namespace msda {

static size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

// false when the shape does not fit the record format (slots and keys are 32-bit: callers split the batch)
bool det_layout(const Dims &d, int value_bytes, DetLayout *out) {
    const long long records = (long long)d.N * d.Lq * d.M * d.L * d.P * 4;
    const long long rows = (long long)d.N * d.S * d.M;
    if (records <= 0 || records > 0x7fffffffLL || rows <= 0 || rows >= 0x7fffffffLL) return false;
    DetLayout l{};
    l.records = records;
    l.rows = (uint32_t)rows;
    l.end_bit = 32 - __builtin_clz(l.rows);
    const size_t r4 = align256((size_t)records * 4);
    l.keys_a = 0;
    l.keys_b = l.keys_a + r4;
    l.ids_a = l.keys_b + r4;
    l.ids_b = l.ids_a + r4;
    l.w = l.ids_b + r4;
    l.start = l.w + align256((size_t)records * value_bytes);
    l.temp = l.start + align256(((size_t)rows + 1) * 4);
    cub::DoubleBuffer<uint32_t> k(nullptr, nullptr), v(nullptr, nullptr);
    size_t tb = 0;
    if (cub::DeviceRadixSort::SortPairs(nullptr, tb, k, v, (int)records, 0, l.end_bit) != cudaSuccess) return false;
    l.temp_bytes = tb;
    l.total = l.temp + align256(tb);
    *out = l;
    return true;
}

DetRecords det_records(void *ws, const DetLayout &l) {
    char *b = static_cast<char *>(ws);
    return DetRecords{reinterpret_cast<uint32_t *>(b + l.keys_a), reinterpret_cast<uint32_t *>(b + l.ids_a),
                      b + l.w, l.rows};
}

namespace {

// start[k] = first sorted record with key >= k, for k in [0, rows]; thread i covers the keys in
// (key[i-1], key[i]] (i == records: up to `rows`, the sentinel)
__global__ void __launch_bounds__(256)
msda_det_bounds_kernel(const uint32_t *__restrict__ keys, long long records, uint32_t rows,
                       uint32_t *__restrict__ start) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i <= records;
         i += (long long)gridDim.x * blockDim.x) {
        const long long prev = i == 0 ? -1 : (long long)keys[i - 1];
        const long long cur = i == records ? (long long)rows : (long long)keys[i];
        for (long long k = prev + 1; k <= cur; ++k) start[k] = (uint32_t)i;
    }
}

// V: element type of grad_output / grad_value (16-bit: widened per term, the row rounded once at the store)
template <typename V, typename T>
__global__ void __launch_bounds__(256)
msda_det_gather_kernel(const uint32_t *__restrict__ start, const uint32_t *__restrict__ ids,
                       const T *__restrict__ w, const V *__restrict__ grad_out, V *__restrict__ grad_value,
                       uint32_t rows, int D, uint32_t rec_per_row) {
    const int lane = threadIdx.x & 31;
    const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
    for (long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); row < rows; row += warps) {
        const uint32_t b = start[row], e = start[row + 1];
        for (int c0 = 0; c0 < D; c0 += 32) {
            const int c = c0 + lane;
            T acc = 0;
            for (uint32_t i0 = b; i0 < e; i0 += 32) {
                // 32 records at a time: lane j fetches record i0 + j, then all lanes walk them in order
                const uint32_t i = i0 + lane;
                uint32_t sl = 0;
                T wl = 0;
                if (i < e) {
                    sl = ids[i];
                    wl = w[sl];
                }
                const uint32_t n = min(32u, e - i0);
#pragma unroll 8
                for (uint32_t j = 0; j < 32; ++j) {
                    if (j < n) {
                        const uint32_t s = __shfl_sync(kFullMask, sl, j);
                        const T ww = __shfl_sync(kFullMask, wl, j);
                        if (c < D) acc = fma_rn(ww, widen<T>(grad_out[(long long)(s / rec_per_row) * D + c]), acc);
                    }
                }
            }
            if (c < D) grad_value[row * D + c] = narrow<V>(acc);
        }
    }
}

unsigned det_grid(long long work, int per_block) {
    long long b = (work + per_block - 1) / per_block;
    const long long cap = (long long)sm_count() * 16;
    if (b > cap) b = cap;
    if (b < 1) b = 1;
    return (unsigned)b;
}

}  // namespace

// Steps 2-4 after the records kernel has filled the workspace.  Counts as three launches
// (msda_b200_launch_count): the sort as one, whatever number of kernels CUB runs for it.
template <typename V, typename T>
cudaError_t launch_det_reduce(const DetLayout &l, void *ws, const V *grad_out, V *grad_value, const Dims &d,
                              cudaStream_t stream) {
    char *b = static_cast<char *>(ws);
    cub::DoubleBuffer<uint32_t> k(reinterpret_cast<uint32_t *>(b + l.keys_a), reinterpret_cast<uint32_t *>(b + l.keys_b));
    cub::DoubleBuffer<uint32_t> v(reinterpret_cast<uint32_t *>(b + l.ids_a), reinterpret_cast<uint32_t *>(b + l.ids_b));
    size_t tb = l.temp_bytes;
    cudaError_t e = cub::DeviceRadixSort::SortPairs(b + l.temp, tb, k, v, (int)l.records, 0, l.end_bit, stream);
    if (e != cudaSuccess) return e;
    note_launch();
    uint32_t *start = reinterpret_cast<uint32_t *>(b + l.start);
    msda_det_bounds_kernel<<<det_grid(l.records + 1, 256), 256, 0, stream>>>(k.Current(), l.records, l.rows, start);
    note_launch();
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    msda_det_gather_kernel<V, T><<<det_grid(l.rows, 8), 256, 0, stream>>>(
        start, v.Current(), reinterpret_cast<const T *>(b + l.w), grad_out, grad_value, l.rows, d.D,
        (uint32_t)(d.L * d.P * 4));
    note_launch();
    return cudaGetLastError();
}

template cudaError_t launch_det_reduce<float, float>(const DetLayout &, void *, const float *, float *, const Dims &,
                                                     cudaStream_t);
template cudaError_t launch_det_reduce<double, double>(const DetLayout &, void *, const double *, double *,
                                                       const Dims &, cudaStream_t);
template cudaError_t launch_det_reduce<__nv_bfloat16, float>(const DetLayout &, void *, const __nv_bfloat16 *,
                                                             __nv_bfloat16 *, const Dims &, cudaStream_t);
template cudaError_t launch_det_reduce<__half, float>(const DetLayout &, void *, const __half *, __half *,
                                                      const Dims &, cudaStream_t);

}  // namespace msda
