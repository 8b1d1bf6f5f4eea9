// scan.cu -- device-wide exclusive prefix sums (reduce / recurse / downsweep).
//
// Used for the small index arrays of the codec (tile counts, radix histograms, compaction flags,
// dictionary offsets).  These arrays are O(rows) or O(uniques) words, a small fraction of the
// TSV bytes; the byte-heavy kernels carry their own decoupled-look-back scans (encode.cu, decode.cu).
#include "common.cuh"

namespace zdwb {

namespace {

constexpr int SCAN_THREADS = 256;
constexpr int SCAN_ITEMS = 8;  // per thread
constexpr int SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

template <typename T>
__global__ void __launch_bounds__(SCAN_THREADS) k_scan_reduce(const T* __restrict__ in, size_t n, T* __restrict__ sums) {
  __shared__ T sh[SCAN_THREADS / 32];
  const size_t base = (size_t)blockIdx.x * SCAN_TILE;
  T acc = 0;
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; ++k) {
    size_t i = base + (size_t)k * SCAN_THREADS + threadIdx.x;
    if (i < n) acc += in[i];
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    T t = 0;
    for (int w = 0; w < SCAN_THREADS / 32; ++w) t += sh[w];
    sums[blockIdx.x] = t;
  }
}

// Each thread owns SCAN_ITEMS consecutive elements (blocked arrangement).
template <typename T>
__global__ void __launch_bounds__(SCAN_THREADS)
    k_scan_down(const T* in, T* out, size_t n, const T* block_offsets, T* total_out) {
  __shared__ T warp_sums[34];
  const size_t base = (size_t)blockIdx.x * SCAN_TILE + (size_t)threadIdx.x * SCAN_ITEMS;
  T v[SCAN_ITEMS];
  T sum = 0;
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; ++k) {
    size_t i = base + k;
    v[k] = i < n ? in[i] : (T)0;
    sum += v[k];
  }
  // block exclusive scan of per-thread sums
  const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  T inc = sum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    T t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= (unsigned)o) inc += t;
  }
  if (lane == 31) warp_sums[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    T w = lane < SCAN_THREADS / 32 ? warp_sums[lane] : (T)0;
    T wi = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      T t = __shfl_up_sync(0xffffffffu, wi, o);
      if (lane >= (unsigned)o) wi += t;
    }
    if (lane < SCAN_THREADS / 32) warp_sums[lane] = wi - w;
    if (lane == 31) warp_sums[32] = wi;
  }
  __syncthreads();
  const T boff = block_offsets ? block_offsets[blockIdx.x] : (T)0;
  T run = boff + warp_sums[warp] + inc - sum;
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; ++k) {
    size_t i = base + k;
    if (i < n) out[i] = run;
    run += v[k];
  }
  if (total_out && blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) *total_out = boff + warp_sums[32];
}

template <typename T>
int exclusive_scan_impl(Ctx* ctx, const T* in, T* out, size_t n, T* total_dev) {
  if (n == 0) {
    if (total_dev) ZDWB_CUDA_TRY(ctx, cudaMemsetAsync(total_dev, 0, sizeof(T), ctx->stream));
    return ZDWB_OK;
  }
  const size_t nb = (n + SCAN_TILE - 1) / SCAN_TILE;
  if (nb == 1) return launch(ctx, "k_scan_down", k_scan_down<T>, 1, SCAN_THREADS, 0, in, out, n, nullptr, total_dev);
  DevBuf sums;
  ZDWB_TRY(sums.alloc(ctx, nb * sizeof(T)));
  ZDWB_TRY(launch(ctx, "k_scan_reduce", k_scan_reduce<T>, (unsigned)nb, SCAN_THREADS, 0, in, n, sums.as<T>()));
  ZDWB_TRY(exclusive_scan_impl<T>(ctx, sums.as<T>(), sums.as<T>(), nb, nullptr));
  return launch(ctx, "k_scan_down", k_scan_down<T>, (unsigned)nb, SCAN_THREADS, 0, in, out, n, sums.as<T>(), total_dev);
}

}  // namespace

int exclusive_scan_u32(Ctx* ctx, const uint32_t* in, uint32_t* out, size_t n, uint32_t* total_dev) {
  return exclusive_scan_impl<uint32_t>(ctx, in, out, n, total_dev);
}
int exclusive_scan_u64(Ctx* ctx, const uint64_t* in, uint64_t* out, size_t n, uint64_t* total_dev) {
  return exclusive_scan_impl<uint64_t>(ctx, in, out, n, total_dev);
}

}  // namespace zdwb
