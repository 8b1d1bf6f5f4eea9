// sort.cu -- orders the unique strings of a block dictionary by strcmp (unsigned bytes, prefix first).
//
// Replaces the red-black tree of the reference (std::map<const char*, ULONG, strcmp-less>,
// dictionary.h:30-35) whose in-order walk defines the on-disk dictionary order (dictionary.cpp:99-108).
//
// Two paths, same result:
//   * small dictionaries (n <= Ctx::small_sort_max, typical for analytics-shaped data): rank by counting over
//     16-byte big-endian prefix keys, all pairs in parallel, ties broken by a byte-wise compare of the remaining bytes;
//   * large dictionaries: LSD radix sort on the 8-byte prefix, then iterative refinement - strings that
//     still tie are re-sorted by (tie-group id, next 8 bytes) until every group is a singleton.  Because
//     the strings are distinct and contain no NUL, zero padding makes "shorter prefix sorts first" fall
//     out of the integer compare.
#include "common.cuh"

namespace zdwb {

namespace {

// ---------------------------------------------------------------------------------------------
// keys
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t prefix_key(const uint8_t* s, uint32_t len, uint32_t off) {
  uint64_t k = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    uint32_t p = off + i;
    uint64_t b = p < len ? (uint64_t)__ldg(s + p) : 0ull;
    k = (k << 8) | b;
  }
  return k;
}

// ids == nullptr -> identity
__global__ void k_make_keys(const uint8_t* __restrict__ base, const uint32_t* __restrict__ starts,
                            const uint32_t* __restrict__ lens, const uint32_t* __restrict__ ids, uint32_t n,
                            uint32_t off, uint64_t* __restrict__ keys, uint32_t* __restrict__ vals_out) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t id = ids ? ids[i] : i;
  keys[i] = prefix_key(base + starts[id], lens[id], off);
  if (vals_out) vals_out[i] = id;
}

// ---------------------------------------------------------------------------------------------
// LSD radix sort of (key u64, seg u32, val u32) records, 8 bits per pass
// ---------------------------------------------------------------------------------------------
constexpr int RS_THREADS = 256;
constexpr int RS_WARPS = RS_THREADS / 32;
// items per thread: 16 for large inputs (few tiles, small histograms), 4 below two million records - a C2-sized dictionary
// (half a million strings) is otherwise 128 CTAs of 16 sequential steps each, on 148 SMs
__host__ __device__ constexpr int rs_tile(int items) { return RS_THREADS * items; }
inline int rs_items_for(const Ctx* ctx, uint32_t n) {
  if (ctx->sort_radix_items == 4 || ctx->sort_radix_items == 16) return (int)ctx->sort_radix_items;  // (tests force either)
  return n < (1u << 21) ? 4 : 16;
}

__device__ __forceinline__ uint32_t rs_digit(const uint64_t* keys, const uint32_t* segs, uint32_t i, int pass) {
  return pass < 8 ? (uint32_t)((keys[i] >> (8 * pass)) & 255u) : ((segs[i] >> (8 * (pass - 8))) & 255u);
}

// One launch per pass ("onesweep"): the digit histogram of the whole record set does not depend on the order of the
// records, so the histograms of all passes of a round are taken in one go up front (k_radix_ghist); a pass's scatter
// then needs, per tile and digit, only the count of that digit in the tiles in front of it - a decoupled look-back over
// per-tile status words.  (The first version ran histogram + three scan launches + scatter per pass: 200 launches for
// a C2-sized dictionary of half a million strings, and the launches were most of the time.)
constexpr int RS_MAX_PASSES = 12;  // 8 key bytes + 4 segment bytes
struct RadixPasses {
  int n;
  int pass[RS_MAX_PASSES];
};
struct RadixScratch {
  uint32_t* ghist;             // [RS_MAX_PASSES][256] digit counts of the round's record set, per pass of the round
  uint32_t* tickets;           // [RS_MAX_PASSES] tiles handed out so far, per pass of the round
  unsigned long long* status;  // [ntiles][256] see os_pack; zeroed once per sort, told apart by the epoch afterwards
  size_t status_bytes;
  uint32_t epoch;              // passes run so far in this sort (never 0 in a status word)
};
constexpr size_t RS_SMALL_BYTES = (size_t)RS_MAX_PASSES * 256 * 4 + 64;  // ghist + tickets: zeroed every round

__global__ void __launch_bounds__(RS_THREADS)
    k_radix_ghist(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ segs, uint32_t n, const RadixPasses P,
                  uint32_t* __restrict__ ghist) {
  __shared__ uint32_t h[RS_MAX_PASSES][256];
  for (int j = threadIdx.x; j < RS_MAX_PASSES * 256; j += RS_THREADS) (&h[0][0])[j] = 0;
  __syncthreads();
  const uint32_t stride = gridDim.x * RS_THREADS;
  const uint32_t rounds = (n + stride - 1) / stride;
  for (uint32_t r = 0; r < rounds; ++r) {  // (whole warps stay together for the vote below)
    const uint32_t i = r * stride + blockIdx.x * RS_THREADS + threadIdx.x;
    const bool valid = i < n;
    const unsigned act = __ballot_sync(0xffffffffu, valid);
    if (!valid) continue;
    const uint64_t k = keys[i];
    const uint32_t sg = segs ? segs[i] : 0u;
    for (int q = 0; q < P.n; ++q) {
      const int pass = P.pass[q];
      const uint32_t d = pass < 8 ? (uint32_t)((k >> (8 * pass)) & 255u) : ((sg >> (8 * (pass - 8))) & 255u);
      // padding bytes and the high bytes of group ids are the same digit for everyone: one add for the warp then
      int same;
      __match_all_sync(act, d, &same);
      if (same) {
        if ((threadIdx.x & 31) == (unsigned)(__ffs(act) - 1)) atomicAdd(&h[q][d], (uint32_t)__popc(act));
      } else {
        atomicAdd(&h[q][d], 1u);
      }
    }
  }
  __syncthreads();
  for (int j = threadIdx.x; j < P.n * 256; j += RS_THREADS) {
    const uint32_t c = (&h[0][0])[j];
    if (c) atomicAdd(ghist + j, c);
  }
}

// status word of (tile, digit): flag (bits 62-63: 1 = the tile's own count, 2 = count of this tile and all in front of
// it) | epoch (bits 40-59) | count (bits 0-39)
__device__ __forceinline__ unsigned long long os_pack(unsigned long long flag, uint32_t epoch, uint32_t count) {
  return (flag << 62) | ((unsigned long long)epoch << 40) | (unsigned long long)count;
}

// Stable scatter of one pass.  Warp w of the CTA owns the contiguous sub-range [tile + w*32*ITEMS, +32*ITEMS) and walks
// it in steps of 32 consecutive items, so the order (warp, step, lane) is the input order.  Tiles are taken in ticket
// order: every tile in front of a running one is running or done, so the look-back cannot wait for a CTA that has not
// started.
template <int RS_ITEMS>
__global__ void __launch_bounds__(RS_THREADS)
    k_radix_onesweep(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ segs, const uint32_t* __restrict__ vals,
                     uint32_t n, int pass, int slot, uint32_t epoch, const uint32_t* __restrict__ ghist,
                     uint32_t* __restrict__ tickets, unsigned long long* status, uint64_t* __restrict__ keys_out,
                     uint32_t* __restrict__ segs_out, uint32_t* __restrict__ vals_out) {
  __shared__ uint32_t wc[RS_WARPS][256];
  __shared__ uint32_t s_tile, s_warp[RS_WARPS];
  const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) s_tile = atomicAdd(tickets + slot, 1u);
  for (int d = lane; d < 256; d += 32) wc[warp][d] = 0;
  __syncthreads();
  const uint32_t tile = s_tile;
  const uint32_t wbase = tile * rs_tile(RS_ITEMS) + warp * (RS_ITEMS * 32);
  // sweep 1: per-warp digit counts
  for (int s = 0; s < RS_ITEMS; ++s) {
    uint32_t i = wbase + s * 32 + lane;
    bool valid = i < n;
    unsigned act = __ballot_sync(0xffffffffu, valid);
    if (valid) {
      uint32_t d = rs_digit(keys, segs, i, pass);
      unsigned peers = __match_any_sync(act, d);
      if (lane == (unsigned)(__ffs(peers) - 1)) wc[warp][d] += __popc(peers);
    }
    __syncwarp();
  }
  __syncthreads();
  {
    const uint32_t d = threadIdx.x;
    uint32_t t = 0;
#pragma unroll
    for (int w = 0; w < RS_WARPS; ++w) t += wc[w][d];
    // ---- records with digit d in the tiles in front of this one
    volatile unsigned long long* st = status + (size_t)tile * 256 + d;
    uint32_t excl = 0;
    if (tile == 0) {
      *st = os_pack(2ull, epoch, t);
    } else {
      *st = os_pack(1ull, epoch, t);
      const volatile unsigned long long* q = status + (size_t)(tile - 1) * 256 + d;
      for (;;) {
        const unsigned long long v = *q;
        if ((uint32_t)((v >> 40) & 0xfffffu) != epoch || (v >> 62) == 0ull) continue;  // not published yet
        excl += (uint32_t)(v & 0xffffffffffull);
        if ((v >> 62) == 2ull) break;
        q -= 256;  // (tile 0 always publishes an inclusive count: the walk ends there at the latest)
      }
      *st = os_pack(2ull, epoch, excl + t);
    }
    // ---- records with a smaller digit: exclusive scan of the pass's global histogram
    const uint32_t g = ghist[slot * 256 + d];
    uint32_t inc = g;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t u = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= (unsigned)o) inc += u;
    }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    uint32_t before = 0;
    for (unsigned w = 0; w < warp; ++w) before += s_warp[w];
    // ---- per digit: global base of this tile, then exclusive over the warps of the CTA
    uint32_t run = before + inc - g + excl;
#pragma unroll
    for (int w = 0; w < RS_WARPS; ++w) {
      uint32_t c = wc[w][d];
      wc[w][d] = run;
      run += c;
    }
  }
  __syncthreads();
  // sweep 2: ranks and scatter
  for (int s = 0; s < RS_ITEMS; ++s) {
    uint32_t i = wbase + s * 32 + lane;
    bool valid = i < n;
    unsigned act = __ballot_sync(0xffffffffu, valid);
    if (valid) {
      uint32_t d = rs_digit(keys, segs, i, pass);
      unsigned peers = __match_any_sync(act, d);
      uint32_t dst = wc[warp][d] + __popc(peers & lanemask_lt());
      __syncwarp(act);
      if (lane == (unsigned)(__ffs(peers) - 1)) wc[warp][d] += __popc(peers);
      keys_out[dst] = keys[i];
      if (segs_out) segs_out[dst] = segs[i];
      vals_out[dst] = vals[i];
    }
    __syncwarp();
  }
}

struct SortBufs {
  uint64_t* key[2];
  uint32_t* seg[2];  // may be null (round 0)
  uint32_t* val[2];
  int cur = 0;
};

// Sorts records [0,n) by digits `pass_list` (least significant first); result ends up in b.{key,seg,val}[b.cur].
int radix_passes(Ctx* ctx, SortBufs& b, uint32_t n, const int* pass_list, int npass, RadixScratch& R) {
  const int items = rs_items_for(ctx, n);
  const uint32_t ntiles = (n + rs_tile(items) - 1) / rs_tile(items);
  if (npass > RS_MAX_PASSES) {
    ctx->err = "sort_strings: too many radix passes in one round";
    return ZDWB_ERR_UNSUPPORTED;
  }
  if (R.epoch + (uint32_t)npass >= (1u << 20)) {  // (a million passes: megabyte-long strings that tie) the epochs start over
    ZDWB_CUDA_TRY(ctx, cudaMemsetAsync(R.status, 0, R.status_bytes, ctx->stream));
    R.epoch = 0;
  }
  RadixPasses P;
  P.n = npass;
  for (int q = 0; q < npass; ++q) P.pass[q] = pass_list[q];
  ZDWB_CUDA_TRY(ctx, cudaMemsetAsync(R.ghist, 0, RS_SMALL_BYTES, ctx->stream));
  const uint32_t grid = std::min<uint32_t>((n + RS_THREADS - 1) / RS_THREADS, (uint32_t)ctx->sm_count * 8);
  ZDWB_TRY(launch(ctx, "k_radix_ghist", k_radix_ghist, grid, RS_THREADS, 0, b.key[b.cur], b.seg[b.cur], n, P, R.ghist));
  for (int q = 0; q < npass; ++q) {
    const int pass = pass_list[q];
    const int s = b.cur, d = b.cur ^ 1;
    const uint32_t epoch = ++R.epoch;
    ZDWB_TRY(launch(ctx, "k_radix_onesweep", items == 4 ? k_radix_onesweep<4> : k_radix_onesweep<16>, ntiles, RS_THREADS, 0,
                    b.key[s], b.seg[s], b.val[s], n, pass, q, epoch, R.ghist, R.tickets, R.status, b.key[d],
                    b.seg[s] ? b.seg[d] : nullptr, b.val[d]));
    b.cur = d;
  }
  return ZDWB_OK;
}

// ---------------------------------------------------------------------------------------------
// refinement bookkeeping
// ---------------------------------------------------------------------------------------------
// head[i] = record i starts a new tie group; unres[i] = record i is in a group of >= 2 records.
__global__ void k_mark_groups(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ segs, uint32_t n,
                              uint32_t* __restrict__ head, uint32_t* __restrict__ unres) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  auto is_head = [&](uint32_t j) -> bool {
    if (j == 0) return true;
    if (keys[j] != keys[j - 1]) return true;
    if (segs && segs[j] != segs[j - 1]) return true;
    return false;
  };
  const bool h = is_head(i);
  const bool next_h = (i + 1 == n) ? true : is_head(i + 1);
  head[i] = h ? 1u : 0u;
  unres[i] = (h && next_h) ? 0u : 1u;
}

// Compacts unresolved records.  pos_in == nullptr -> identity (round 0).
__global__ void k_compact_unresolved(const uint32_t* __restrict__ unres, const uint32_t* __restrict__ unres_scan,
                                     const uint32_t* __restrict__ head_scan, const uint32_t* __restrict__ vals,
                                     const uint32_t* __restrict__ pos_in, uint32_t n, uint32_t* __restrict__ ids_out,
                                     uint32_t* __restrict__ seg_out, uint32_t* __restrict__ pos_out) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || !unres[i]) return;
  const uint32_t j = unres_scan[i];
  ids_out[j] = vals[i];
  seg_out[j] = head_scan[i];  // group id = (#heads in [0..i]) - 1, prepared by k_group_ids
  pos_out[j] = pos_in ? pos_in[i] : i;
}

// group id of record i = (#heads in [0..i]) - 1, from the exclusive scan of head[]
__global__ void k_group_ids(const uint32_t* __restrict__ head, uint32_t* __restrict__ head_scan, uint32_t n) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  head_scan[i] = head_scan[i] + head[i] - 1u;
}

__global__ void k_scatter_order(const uint32_t* __restrict__ pos, const uint32_t* __restrict__ vals, uint32_t n,
                                uint32_t* __restrict__ order) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) order[pos[i]] = vals[i];
}

// ---------------------------------------------------------------------------------------------
// small path: rank by counting.  rank(i) = #{ j : s_j < s_i } = sum over tiles of 1024 strings of the lower bound of
// s_i's 16-byte big-endian prefix key among the tile's sorted keys (bitonic sort in shared memory, then one binary
// search per string and tile); only strings whose prefixes tie fall back to the bytes in memory.  n^2 / 100 key
// compares spread over the whole GPU, three launches, no multi-pass radix machinery.
// ---------------------------------------------------------------------------------------------
constexpr int RK_THREADS = 256;
constexpr int RK_JTILE = 1024;

// four bytes at an arbitrary address, all of them inside the buffer (only aligned words that hold one of them are read)
__device__ __forceinline__ uint32_t load4_unaligned(const uint8_t* p) {
  const uintptr_t a = reinterpret_cast<uintptr_t>(p);
  const uint32_t* w = reinterpret_cast<const uint32_t*>(a & ~(uintptr_t)3);
  const uint32_t sh = (uint32_t)(a & 3u) * 8u;
  const uint32_t lo = __ldg(w), hi = sh ? __ldg(w + 1) : 0u;
  return __funnelshift_r(lo, hi, sh);
}

// strcmp order of two strings that agree on their first `from` bytes: sixteen bytes a round (the eight loads of a round
// are in flight together - the compares of a tie group are a chain of dependent rounds, so the round count is what
// counts), words compared as big-endian numbers (= unsigned byte order), then the tail; a proper prefix sorts first
__device__ __forceinline__ bool str_less_from(const uint8_t* base, uint32_t sa, uint32_t la, uint32_t sb, uint32_t lb,
                                              uint32_t from) {
  const uint32_t m = la < lb ? la : lb;
  uint32_t i = from;
  if (i + 16 <= m) {
    const uintptr_t ua = reinterpret_cast<uintptr_t>(base + sa + i), ub = reinterpret_cast<uintptr_t>(base + sb + i);
    const uint32_t* wa = reinterpret_cast<const uint32_t*>(ua & ~(uintptr_t)3);
    const uint32_t* wb = reinterpret_cast<const uint32_t*>(ub & ~(uintptr_t)3);
    const uint32_t sha = (uint32_t)(ua & 3u) * 8u, shb = (uint32_t)(ub & 3u) * 8u;
    // (only aligned words that hold one of the round's 16 bytes are read: five when the side is shifted, else four)
    for (; i + 16 <= m; i += 16, wa += 4, wb += 4) {
      const uint32_t a0 = __ldg(wa), a1 = __ldg(wa + 1), a2 = __ldg(wa + 2), a3 = __ldg(wa + 3), a4 = sha ? __ldg(wa + 4) : 0u;
      const uint32_t b0 = __ldg(wb), b1 = __ldg(wb + 1), b2 = __ldg(wb + 2), b3 = __ldg(wb + 3), b4 = shb ? __ldg(wb + 4) : 0u;
      const uint32_t x0 = __funnelshift_r(a0, a1, sha), y0 = __funnelshift_r(b0, b1, shb);
      const uint32_t x1 = __funnelshift_r(a1, a2, sha), y1 = __funnelshift_r(b1, b2, shb);
      const uint32_t x2 = __funnelshift_r(a2, a3, sha), y2 = __funnelshift_r(b2, b3, shb);
      const uint32_t x3 = __funnelshift_r(a3, a4, sha), y3 = __funnelshift_r(b3, b4, shb);
      if (x0 != y0) return __byte_perm(x0, 0, 0x0123) < __byte_perm(y0, 0, 0x0123);
      if (x1 != y1) return __byte_perm(x1, 0, 0x0123) < __byte_perm(y1, 0, 0x0123);
      if (x2 != y2) return __byte_perm(x2, 0, 0x0123) < __byte_perm(y2, 0, 0x0123);
      if (x3 != y3) return __byte_perm(x3, 0, 0x0123) < __byte_perm(y3, 0, 0x0123);
    }
  }
  for (; i + 4 <= m; i += 4) {
    const uint32_t a = load4_unaligned(base + sa + i), b = load4_unaligned(base + sb + i);
    if (a != b) return __byte_perm(a, 0, 0x0123) < __byte_perm(b, 0, 0x0123);
  }
  for (; i < m; ++i) {
    const uint8_t a = __ldg(base + sa + i), b = __ldg(base + sb + i);
    if (a != b) return a < b;
  }
  return la < lb;
}

__global__ void k_rank_keys(const uint8_t* __restrict__ base, const uint32_t* __restrict__ starts,
                            const uint32_t* __restrict__ lens, uint32_t n, ulonglong2* __restrict__ keys) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint8_t* s = base + starts[i];
  const uint32_t len = lens[i];
  keys[i] = make_ulonglong2(prefix_key(s, len, 0), prefix_key(s, len, 8));
}

// (x, y) as one 128-bit big number
__device__ __forceinline__ bool key_less(const ulonglong2& a, const ulonglong2& b) { return a.x < b.x || (a.x == b.x && a.y < b.y); }

// Sorts every tile of RK_JTILE prefix keys (with the string ids as payload) in shared memory: bitonic network, one
// compare-exchange per thread and stage.  Short tiles are padded with (max key, max id), which sort behind everything.
constexpr int RK_SORT_THREADS = RK_JTILE / 2;
__global__ void __launch_bounds__(RK_SORT_THREADS)
    k_rank_tile_sort(const ulonglong2* __restrict__ keys, uint32_t n, ulonglong2* __restrict__ skeys, uint32_t* __restrict__ sidx) {
  __shared__ ulonglong2 k[RK_JTILE];
  __shared__ uint32_t id[RK_JTILE];
  const uint32_t j0 = blockIdx.x * RK_JTILE;
  for (uint32_t t = threadIdx.x; t < RK_JTILE; t += RK_SORT_THREADS) {
    const uint32_t g = j0 + t;
    k[t] = g < n ? keys[g] : make_ulonglong2(~0ull, ~0ull);
    id[t] = g < n ? g : 0xffffffffu;
  }
  __syncthreads();
  for (uint32_t size = 2; size <= RK_JTILE; size <<= 1) {
    for (uint32_t stride = size >> 1; stride > 0; stride >>= 1) {
      const uint32_t t = threadIdx.x;
      const uint32_t lo = 2u * t - (t & (stride - 1u)), hi = lo + stride;
      const bool asc = (lo & size) == 0u;
      const ulonglong2 a = k[lo], b = k[hi];
      const uint32_t ia = id[lo], ib = id[hi];
      const bool a_gt_b = key_less(b, a) || (!key_less(a, b) && ia > ib);
      if (a_gt_b == asc) {
        k[lo] = b;
        k[hi] = a;
        id[lo] = ib;
        id[hi] = ia;
      }
      __syncthreads();
    }
  }
  for (uint32_t t = threadIdx.x; t < RK_JTILE; t += RK_SORT_THREADS) {
    const uint32_t g = j0 + t;
    if (g < n) {
      skeys[g] = k[t];
      sidx[g] = id[t];
    }
  }
}

// rank(i) += #{ j in tile : s_j < s_i }: lower bound of key_i among the tile's sorted keys; the strings that agree
// with s_i on all 16 prefix bytes (a run right at the lower bound) are compared in memory.
// strings per thread: 1 for small sets (a tie group is a serial chain of string compares: spread them), 4 for large
// ones (every CTA first copies its tile of keys into shared memory)
__global__ void __launch_bounds__(RK_THREADS)
    k_rank_count(const uint8_t* __restrict__ base, const uint32_t* __restrict__ starts, const uint32_t* __restrict__ lens,
                 const ulonglong2* __restrict__ keys, const ulonglong2* __restrict__ skeys, const uint32_t* __restrict__ sidx,
                 uint32_t n, uint32_t ipt, uint32_t* __restrict__ rank) {
  __shared__ ulonglong2 sk[RK_JTILE];
  const uint32_t j0 = blockIdx.y * RK_JTILE, jn = min((uint32_t)RK_JTILE, n - j0);
  for (uint32_t t = threadIdx.x; t < jn; t += RK_THREADS) sk[t] = skeys[j0 + t];
  __syncthreads();
#pragma unroll 1
  for (uint32_t r = 0; r < ipt; ++r) {
    const uint32_t i = (blockIdx.x * ipt + r) * RK_THREADS + threadIdx.x;
    if (i >= n) break;
    const ulonglong2 me = keys[i];
    uint32_t lo = 0, hi = jn;
    while (lo < hi) {
      const uint32_t m = (lo + hi) >> 1;
      if (key_less(sk[m], me)) lo = m + 1;
      else hi = m;
    }
    uint32_t cnt = lo;
    for (uint32_t t = lo; t < jn; ++t) {
      const ulonglong2 o = sk[t];
      if (o.x != me.x || o.y != me.y) break;
      const uint32_t j = sidx[j0 + t];
      if (j != i && str_less_from(base, starts[j], lens[j], starts[i], lens[i], 16)) ++cnt;
    }
    if (cnt) atomicAdd(rank + i, cnt);
  }
}

__global__ void k_rank_scatter(const uint32_t* __restrict__ rank, uint32_t n, uint32_t* __restrict__ order) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) order[rank[i]] = i;
}

}  // namespace

int sort_strings(Ctx* ctx, const uint8_t* base, const uint32_t* starts, const uint32_t* lens, uint32_t n,
                 uint32_t max_len, uint32_t* order_out) {
  if (n == 0) return ZDWB_OK;
  cudaStream_t st = ctx->stream;

  // ---- small path
  long long small_max = ctx->small_sort_max;
  if (small_max > (1 << 20)) small_max = 1 << 20;
  if ((long long)n <= small_max) {
    DevBuf keys, rank, skeys, sidx;
    ZDWB_TRY(keys.alloc(ctx, (size_t)n * sizeof(ulonglong2)));
    ZDWB_TRY(skeys.alloc(ctx, (size_t)n * sizeof(ulonglong2)));
    ZDWB_TRY(sidx.alloc(ctx, (size_t)n * 4));
    ZDWB_TRY(rank.alloc(ctx, (size_t)n * 4));
    ZDWB_CUDA_TRY(ctx, cudaMemsetAsync(rank.p, 0, (size_t)n * 4, st));
    const unsigned gi = (n + RK_THREADS - 1) / RK_THREADS, ntile = (n + RK_JTILE - 1) / RK_JTILE;
    ZDWB_TRY(launch(ctx, "k_rank_keys", k_rank_keys, gi, RK_THREADS, 0, base, starts, lens, n, keys.as<ulonglong2>()));
    ZDWB_TRY(launch(ctx, "k_rank_tile_sort", k_rank_tile_sort, ntile, RK_SORT_THREADS, 0, keys.as<ulonglong2>(), n,
                    skeys.as<ulonglong2>(), sidx.as<uint32_t>()));
    const uint32_t ipt = n > 16384 ? 4 : 1;
    ZDWB_TRY(launch(ctx, "k_rank_count", k_rank_count, dim3((gi + ipt - 1) / ipt, ntile), RK_THREADS, 0, base, starts, lens,
                    keys.as<ulonglong2>(), skeys.as<ulonglong2>(), sidx.as<uint32_t>(), n, ipt, rank.as<uint32_t>()));
    return launch(ctx, "k_rank_scatter", k_rank_scatter, gi, RK_THREADS, 0, rank.as<uint32_t>(), n, order_out);
  }

  // ---- large path
  // refinement rounds sort m <= n records and may pick the smaller tile: size the status words for the worst of the two
  const uint32_t ntiles = std::max<uint32_t>((n + rs_tile(rs_items_for(ctx, n)) - 1) / rs_tile(rs_items_for(ctx, n)),
                                             (std::min<uint32_t>(n, 1u << 21) + rs_tile(4) - 1) / rs_tile(4));
  DevBuf keyA, keyB, segA, segB, valA, valB, hist, head, unres, unres_scan, ids, pos, pos2, total;
  ZDWB_TRY(keyA.alloc(ctx, (size_t)n * 8));
  ZDWB_TRY(keyB.alloc(ctx, (size_t)n * 8));
  ZDWB_TRY(valA.alloc(ctx, (size_t)n * 4));
  ZDWB_TRY(valB.alloc(ctx, (size_t)n * 4));
  ZDWB_TRY(hist.alloc(ctx, RS_SMALL_BYTES + (size_t)ntiles * 256 * 8));
  ZDWB_CUDA_TRY(ctx, cudaMemsetAsync(hist.p, 0, RS_SMALL_BYTES + (size_t)ntiles * 256 * 8, st));
  RadixScratch RSc;
  RSc.ghist = hist.as<uint32_t>();
  RSc.tickets = RSc.ghist + RS_MAX_PASSES * 256;
  RSc.status = reinterpret_cast<unsigned long long*>(reinterpret_cast<uint8_t*>(hist.p) + RS_SMALL_BYTES);
  RSc.status_bytes = (size_t)ntiles * 256 * 8;
  RSc.epoch = 0;
  ZDWB_TRY(head.alloc(ctx, (size_t)n * 4));
  ZDWB_TRY(unres.alloc(ctx, (size_t)n * 4));
  ZDWB_TRY(unres_scan.alloc(ctx, (size_t)n * 4));
  ZDWB_TRY(total.alloc(ctx, 16));

  const unsigned g256 = (n + 255) / 256;
  SortBufs b;
  b.key[0] = keyA.as<uint64_t>();
  b.key[1] = keyB.as<uint64_t>();
  b.seg[0] = b.seg[1] = nullptr;
  b.val[0] = valA.as<uint32_t>();
  b.val[1] = valB.as<uint32_t>();
  b.cur = 0;

  // round 0: sort everything by the first 8 bytes
  ZDWB_TRY(launch(ctx, "k_make_keys", k_make_keys, g256, 256, 0, base, starts, lens, nullptr, n, 0, b.key[0], b.val[0]));
  {
    const int passes[8] = {0, 1, 2, 3, 4, 5, 6, 7};
    ZDWB_TRY(radix_passes(ctx, b, n, passes, 8, RSc));
  }
  ZDWB_CUDA_TRY(ctx, cudaMemcpyAsync(order_out, b.val[b.cur], (size_t)n * 4, cudaMemcpyDeviceToDevice, st));

  // tie groups of round 0
  ZDWB_TRY(launch(ctx, "k_mark_groups", k_mark_groups, g256, 256, 0, b.key[b.cur], nullptr, n, head.as<uint32_t>(),
                  unres.as<uint32_t>()));
  ZDWB_TRY(exclusive_scan_u32(ctx, unres.as<uint32_t>(), unres_scan.as<uint32_t>(), n, total.as<uint32_t>()));
  uint32_t m = 0;
  ZDWB_CUDA_TRY(ctx, cudaMemcpyAsync(ctx->meta_host, total.p, 4, cudaMemcpyDeviceToHost, st));
  ZDWB_CUDA_TRY(ctx, cudaStreamSynchronize(st));
  m = *reinterpret_cast<uint32_t*>(ctx->meta_host);
  if (m == 0) return ZDWB_OK;

  // unresolved records: ids, group ids, target positions
  ZDWB_TRY(segA.alloc(ctx, (size_t)m * 4));
  ZDWB_TRY(segB.alloc(ctx, (size_t)m * 4));
  ZDWB_TRY(ids.alloc(ctx, (size_t)m * 4));
  ZDWB_TRY(pos.alloc(ctx, (size_t)m * 4));
  ZDWB_TRY(pos2.alloc(ctx, (size_t)m * 4));
  {
    DevBuf head_scan;
    ZDWB_TRY(head_scan.alloc(ctx, (size_t)n * 4));
    ZDWB_TRY(exclusive_scan_u32(ctx, head.as<uint32_t>(), head_scan.as<uint32_t>(), n, nullptr));
    ZDWB_TRY(launch(ctx, "k_group_ids", k_group_ids, g256, 256, 0, head.as<uint32_t>(), head_scan.as<uint32_t>(), n));
    ZDWB_TRY(launch(ctx, "k_compact_unresolved", k_compact_unresolved, g256, 256, 0, unres.as<uint32_t>(), unres_scan.as<uint32_t>(),
                    head_scan.as<uint32_t>(), b.val[b.cur], nullptr, n, ids.as<uint32_t>(), segA.as<uint32_t>(), pos.as<uint32_t>()));
  }
  uint32_t* pos_cur = pos.as<uint32_t>();
  uint32_t* pos_nxt = pos2.as<uint32_t>();
  // group ids are numbered over the record set they were computed on: all n records after round 0,
  // the previous round's m records afterwards
  uint32_t seg_max = n - 1;

  for (uint32_t round = 1;; ++round) {
    const uint32_t off = round * 8;
    if (off > max_len + 8) {
      ctx->err = "sort_strings: tie groups did not resolve (duplicate strings in the unique set?)";
      return ZDWB_ERR_CUDA;
    }
    const unsigned gm = (m + 255) / 256;
    // records: key = next 8 bytes, seg = group id, val = string id
    b.seg[0] = segA.as<uint32_t>();
    b.seg[1] = segB.as<uint32_t>();
    // the current group ids live in segA; make sure the record set starts in slot 0
    b.cur = 0;
    ZDWB_TRY(launch(ctx, "k_make_keys", k_make_keys, gm, 256, 0, base, starts, lens, ids.as<uint32_t>(), m, off, b.key[0], b.val[0]));
    int passes[12];
    int np = 0;
    for (int p = 0; p < 8; ++p) passes[np++] = p;
    const uint32_t seg_bytes = bytes_needed((uint64_t)seg_max);
    for (uint32_t p = 0; p < seg_bytes; ++p) passes[np++] = 8 + (int)p;
    ZDWB_TRY(radix_passes(ctx, b, m, passes, np, RSc));
    // write the refined order back to the positions these records occupy
    ZDWB_TRY(launch(ctx, "k_scatter_order", k_scatter_order, gm, 256, 0, pos_cur, b.val[b.cur], m, order_out));
    // new tie groups
    ZDWB_TRY(launch(ctx, "k_mark_groups", k_mark_groups, gm, 256, 0, b.key[b.cur], b.seg[b.cur], m, head.as<uint32_t>(),
                    unres.as<uint32_t>()));
    ZDWB_TRY(exclusive_scan_u32(ctx, unres.as<uint32_t>(), unres_scan.as<uint32_t>(), m, total.as<uint32_t>()));
    ZDWB_CUDA_TRY(ctx, cudaMemcpyAsync(ctx->meta_host, total.p, 4, cudaMemcpyDeviceToHost, st));
    ZDWB_CUDA_TRY(ctx, cudaStreamSynchronize(st));
    const uint32_t m2 = *reinterpret_cast<uint32_t*>(ctx->meta_host);
    if (m2 == 0) break;
    {
      DevBuf head_scan;
      ZDWB_TRY(head_scan.alloc(ctx, (size_t)m * 4));
      ZDWB_TRY(exclusive_scan_u32(ctx, head.as<uint32_t>(), head_scan.as<uint32_t>(), m, nullptr));
      ZDWB_TRY(launch(ctx, "k_group_ids", k_group_ids, gm, 256, 0, head.as<uint32_t>(), head_scan.as<uint32_t>(), m));
      // compact into (ids, segA, pos_nxt).  The kernel reads none of the seg arrays (k_mark_groups, the last
      // reader of the sorted segs, is already ordered before it), so the new group ids go straight to segA.
      ZDWB_TRY(launch(ctx, "k_compact_unresolved", k_compact_unresolved, gm, 256, 0, unres.as<uint32_t>(), unres_scan.as<uint32_t>(),
                      head_scan.as<uint32_t>(), b.val[b.cur], pos_cur, m, ids.as<uint32_t>(), segA.as<uint32_t>(), pos_nxt));
    }
    uint32_t* t = pos_cur;
    pos_cur = pos_nxt;
    pos_nxt = t;
    seg_max = m - 1;
    m = m2;
  }
  return ZDWB_OK;
}

}  // namespace zdwb
