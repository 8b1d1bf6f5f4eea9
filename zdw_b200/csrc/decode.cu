// decode.cu -- one ZDW block -> TSV rows, entirely on the GPU.
//
// Replaces UnconvertFromZDW_Base::parseBlockHeader (UnconvertFromZDW.cpp:758-1000) and the per-row loop
// UnconvertFromZDW<T>::readNextRow (:1270-1464) with GetWord (:359-371), llutoa/lltoa (:318-356) and
// outputDefault (:1224-1266).
//
// The encoded row stream has no row lengths: a row is ceil(U/8) flag bytes followed by the values of the
// flagged columns, so where row r+1 starts is only known after row r's flags have been read.  The kernels:
//   k_dec_tile_maps    for every tile of the stream and every possible entry offset e in [0, M) (M = max row
//                      bytes): where does a walk that enters the tile at e leave it, and how many rows start
//                      inside?  Row length at a byte position is a popcount over 4 size bit-planes.
//   k_dec_compose      composes those maps group by group (function composition is associative) ...
//   k_dec_descend      ... and hands every tile its true entry offset and first row number.
//   k_dec_row_starts   one group of lanes per tile walks the true chain and records row_off[r].
//   k_dec_strip_summary / k_carry_*   last explicit value per (strip of rows, used column) and its
//                      propagation across strips: the value a column holds where a strip begins.
//   k_dec_rows<false>  (k_dec_row_lens) one group of lanes per strip walks its rows keeping the text length of every
//                      output item: row lengths -> exclusive scan -> row offsets and the exact output size.
//   k_dec_rows<true>   (k_dec_write_rows) the same walk with the rendered texts kept in shared memory; every row is
//                      assembled straight in global memory from a static template and the items' texts.
// The row-walking kernels give a row to 32 lanes, or to 16 / 8 when the schema is narrow (several rows per warp).
// zdwb_decode_columns shares the row-boundary discovery and the carries (strips of 32 rows), then
//   k_dict_counts / k_dict_entries   where every dictionary entry starts (a scan over the NUL map's popcounts), so that a
//                      text offset becomes the entry's rank (its code) in O(1)
//   k_dec_columns      one warp per strip, one lane per row: the int64 of every selected column in every row.
#include <algorithm>
#include <deque>
#include <string>
#include <type_traits>
#include <vector>

#include "common.cuh"
#include "carry.cuh"

namespace zdwb {

namespace {

constexpr int DEC_THREADS = 256;
constexpr int DEC_WARPS = DEC_THREADS / 32;

struct DecMeta {
  uint32_t err;            // 1 = dictionary offset out of range (CORRUPTED_DATA_ERROR)
  uint32_t tile_ticket;
  unsigned long long out_bytes;
  uint32_t overflow;       // output buffer estimate too small
  uint32_t pad;
};

struct DecParams {
  const uint8_t* blk;   // device pointer to the block (numRows field)
  uint64_t avail;       // bytes readable from blk
  uint64_t rows_base;   // offset of the first encoded row
  uint64_t dict_base;   // offset of the dictionary origin byte
  uint64_t dict_total;  // dictionary bytes incl. the origin byte
  uint32_t nrows, U, F, M, W;
  const uint8_t* usz;          // [U] value width of every used column
  const unsigned long long* ubase;  // [U]
  const uint8_t* utype;        // [U]
  const uint32_t* planes;      // [4][W] bit k of the width of used column u, as flag-word masks
  const uint32_t* nulmap;      // bit i = dictionary byte i is NUL (one all-ones word appended): entry lengths in O(1)
};

__device__ __forceinline__ uint32_t stream_byte(const DecParams& P, uint64_t s) {
  const uint64_t a = P.rows_base + s;
  return a < P.avail ? (uint32_t)__ldg(P.blk + a) : 0u;
}

// ---------------------------------------------------------------------------------------------
// row-boundary discovery
// ---------------------------------------------------------------------------------------------
// maps[tile*M + e] = (rows started << 32) | exit offset into the next tile
__global__ void __launch_bounds__(DEC_THREADS)
    k_dec_tile_maps(const DecParams P, uint64_t win_bytes, uint32_t T, uint64_t* __restrict__ maps) {
  extern __shared__ __align__(16) uint8_t dsm[];
  // layout: next[T] u32 | words[(T + 4W + 8)/4] u32 | planes[4W] u32
  uint32_t* next = reinterpret_cast<uint32_t*>(dsm);
  uint32_t* words = next + T;
  const uint32_t nwords = (T + 4 * P.W + 8) / 4;
  uint32_t* planes = words + nwords;
  const uint64_t t0 = (uint64_t)blockIdx.x * T;
  for (uint32_t i = threadIdx.x; i < nwords; i += DEC_THREADS) {
    uint32_t w = 0;
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      const uint64_t s = t0 + (uint64_t)i * 4 + b;
      const uint32_t v = s < win_bytes ? stream_byte(P, s) : 0u;
      w |= v << (8 * b);
    }
    words[i] = w;
  }
  for (uint32_t i = threadIdx.x; i < 4 * P.W; i += DEC_THREADS) planes[i] = P.planes[i];
  __syncthreads();
  const uint32_t W = P.W;
  if (W <= 8) {
    // up to 256 used columns: the bit planes stay in registers for all of the thread's positions
    uint32_t pl[4][8];
#pragma unroll
    for (int w = 0; w < 8; ++w) {
#pragma unroll
      for (int k = 0; k < 4; ++k) pl[k][w] = (uint32_t)w < W ? planes[k * W + w] : 0u;
    }
    for (uint32_t s = threadIdx.x; s < T; s += DEC_THREADS) {
      const uint32_t a = s >> 2, sh = (s & 3u) * 8u;
      uint32_t prev = words[a];
      uint32_t acc = P.F;
#pragma unroll
      for (int w = 0; w < 8; ++w) {
        if ((uint32_t)w < W) {
          const uint32_t nxt = words[a + w + 1];
          const uint32_t word = __funnelshift_r(prev, nxt, sh);
          prev = nxt;
          acc += __popc(word & pl[0][w]) + 2u * __popc(word & pl[1][w]) + 4u * __popc(word & pl[2][w]) + 8u * __popc(word & pl[3][w]);
        }
      }
      next[s] = s + acc;
    }
  } else {
    for (uint32_t s = threadIdx.x; s < T; s += DEC_THREADS) {
      const uint32_t a = s >> 2, sh = (s & 3u) * 8u;
      uint32_t prev = words[a];
      uint32_t acc = P.F;
      for (uint32_t w = 0; w < W; ++w) {
        const uint32_t nxt = words[a + w + 1];
        const uint32_t word = __funnelshift_r(prev, nxt, sh);
        prev = nxt;
        acc += __popc(word & planes[w]) + 2u * __popc(word & planes[W + w]) + 4u * __popc(word & planes[2 * W + w]) +
               8u * __popc(word & planes[3 * W + w]);
      }
      next[s] = s + acc;
    }
  }
  __syncthreads();
  for (uint32_t e = threadIdx.x; e < P.M; e += DEC_THREADS) {
    uint32_t p = e, c = 0;
    while (p < T) {
      p = next[p];
      ++c;
    }
    maps[(size_t)blockIdx.x * P.M + e] = ((uint64_t)c << 32) | (uint64_t)(p - T);
  }
}

// out[g][e] = in[gG + G-1] o ... o in[gG] (e)
__global__ void __launch_bounds__(DEC_THREADS)
    k_dec_compose(const uint64_t* __restrict__ in, uint32_t n_in, uint32_t M, uint32_t G, uint64_t* __restrict__ out) {
  const uint32_t g = blockIdx.x;
  const uint32_t tb = g * G, te = min(n_in, tb + G);
  for (uint32_t e = threadIdx.x; e < M; e += DEC_THREADS) {
    uint32_t x = e;
    uint32_t c = 0;
    for (uint32_t t = tb; t < te; ++t) {
      const uint64_t v = in[(size_t)t * M + x];
      x = (uint32_t)v;
      c += (uint32_t)(v >> 32);
    }
    out[(size_t)g * M + e] = ((uint64_t)c << 32) | x;
  }
}

// ent_child[t] = state on entering child t: (rows before << 32) | entry offset
__global__ void k_dec_descend(const uint64_t* __restrict__ in, uint32_t n_in, uint32_t M, uint32_t G,
                              const uint64_t* __restrict__ ent_parent, uint32_t n_parent, uint64_t* __restrict__ ent_child) {
  const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n_parent) return;
  uint64_t st = ent_parent[g];
  const uint32_t tb = g * G, te = min(n_in, tb + G);
  for (uint32_t t = tb; t < te; ++t) {
    ent_child[t] = st;
    const uint64_t v = in[(size_t)t * M + (uint32_t)st];
    st = (((st >> 32) + (v >> 32)) << 32) | (uint32_t)v;
  }
}

// row length at stream offset p, worked out by the GL lanes of a group (GL = 32: the whole warp)
template <int GL>
__device__ __forceinline__ uint32_t group_row_len(const DecParams& P, uint64_t p) {
  const unsigned gl = lane_id() & (unsigned)(GL - 1);
  const unsigned gm = GL == 32 ? 0xffffffffu : (((1u << GL) - 1u) << (lane_id() & ~(unsigned)(GL - 1)));
  uint32_t acc = 0;
  for (uint32_t w0 = 0; w0 < P.W; w0 += GL) {
    const uint32_t w = w0 + gl;
    if (w < P.W) {
      uint32_t word = 0;
#pragma unroll
      for (int b = 0; b < 4; ++b) word |= stream_byte(P, p + 4ull * w + b) << (8 * b);
      acc += __popc(word & P.planes[w]) + 2u * __popc(word & P.planes[P.W + w]) +
             4u * __popc(word & P.planes[2 * P.W + w]) + 8u * __popc(word & P.planes[3 * P.W + w]);
    }
  }
#pragma unroll
  for (int o = GL / 2; o > 0; o >>= 1) acc += __shfl_xor_sync(gm, acc, o, GL);
  return P.F + acc;
}

// one group of GL lanes per tile walks the true chain of rows and records row_off[r]
template <int GL>
__global__ void __launch_bounds__(DEC_THREADS)
    k_dec_row_starts(const DecParams P, uint32_t T, uint32_t ntiles, const uint64_t* __restrict__ ent,
                     uint32_t* __restrict__ row_off) {
  const uint32_t tile = (blockIdx.x * DEC_WARPS + (threadIdx.x >> 5)) * (32 / GL) + lane_id() / GL;
  if (tile >= ntiles) return;
  const uint64_t st = ent[tile];
  uint64_t r = st >> 32;
  uint64_t p = (uint64_t)tile * T + (uint32_t)st;
  const uint64_t pend = (uint64_t)(tile + 1) * T;
  while (p < pend && r <= P.nrows) {
    if ((lane_id() & (unsigned)(GL - 1)) == 0) row_off[r] = (uint32_t)p;
    if (r == P.nrows) break;
    p += group_row_len<GL>(P, p);
    ++r;
  }
}

// ---------------------------------------------------------------------------------------------
// row parser: one warp walks the flag bytes of a row and calls cb(u, value offset inside the row)
// for every flagged used column, lanes working on different flag bytes.  `planes` = the 4 bit planes of the
// column widths (shared or global memory): the value bytes selected by flag byte j are
// sum_k 2^k * popc(flags & plane_k byte j).
// ---------------------------------------------------------------------------------------------
// A group of G consecutive lanes (G = 32: the whole warp; 8 or 16: narrow schemas, several rows per warp) works on one
// row.  group_mask = the lanes of the caller's group, for the *_sync primitives.
template <int G>
__device__ __forceinline__ unsigned group_mask() {
  return G == 32 ? 0xffffffffu : (((1u << G) - 1u) << (lane_id() & ~(unsigned)(G - 1)));
}

// `fb0` = the flag byte of group lane j for the first round (j < F), loaded ahead of time by the caller.
template <int G, class CB>
__device__ __forceinline__ void warp_parse_row(const DecParams& P, const uint32_t* __restrict__ planes,
                                               const uint8_t* __restrict__ rp, uint32_t fb0, CB&& cb) {
  const unsigned gl = lane_id() & (unsigned)(G - 1), gm = group_mask<G>();
  uint32_t run = P.F;
  for (uint32_t j0 = 0; j0 < P.F; j0 += G) {
    const uint32_t j = j0 + gl;
    uint32_t fb = 0, bl = 0;
    if (j < P.F) {
      fb = j0 ? (uint32_t)__ldg(rp + j) : fb0;
      if (fb) {
        const uint32_t sh = (j & 3u) * 8u, w = j >> 2;
        bl = __popc(fb & (planes[w] >> sh)) + 2u * __popc(fb & (planes[P.W + w] >> sh)) +
             4u * __popc(fb & (planes[2 * P.W + w] >> sh)) + 8u * __popc(fb & (planes[3 * P.W + w] >> sh));
      }
    }
    uint32_t inc = bl;
#pragma unroll
    for (int o = 1; o < G; o <<= 1) {
      uint32_t t = __shfl_up_sync(gm, inc, o, G);
      if (gl >= (unsigned)o) inc += t;
    }
    const uint32_t tot = __shfl_sync(gm, inc, G - 1, G);
    uint32_t voff = run + inc - bl;
    while (fb) {
      const int b = __ffs(fb) - 1;
      fb &= fb - 1;
      const uint32_t u = j * 8 + b;
      if (u < P.U) {
        cb(u, voff);
        voff += P.usz[u];
      }
    }
    run += tot;
  }
}
template <int G>
__device__ __forceinline__ uint32_t first_flag_byte(const DecParams& P, const uint8_t* __restrict__ rp) {
  const unsigned gl = lane_id() & (unsigned)(G - 1);
  return gl < P.F ? (uint32_t)__ldg(rp + gl) : 0u;
}

// little-endian value of sz (1..8) bytes at an arbitrary address: two aligned 64-bit loads
__device__ __forceinline__ unsigned long long load_le(const uint8_t* __restrict__ p, uint32_t sz) {
  const uintptr_t a = reinterpret_cast<uintptr_t>(p);
  const unsigned long long* w = reinterpret_cast<const unsigned long long*>(a & ~(uintptr_t)7);
  const uint32_t sh = (uint32_t)(a & 7u) * 8u;
  unsigned long long v = __ldg(w) >> sh;
  if (sh + sz * 8u > 64u) v |= __ldg(w + 1) << (64u - sh);
  return sz >= 8 ? v : (v & ((1ull << (sz * 8u)) - 1ull));
}

// last explicit value of every used column inside a strip of R rows; optionally (-t / -s) bounds-checks the
// dictionary offset of every explicit value (UnconvertFromZDW.cpp:1527-1560) and counts the set flag bits per column
template <int GL>
__global__ void __launch_bounds__(DEC_THREADS)
    k_dec_strip_summary(const DecParams P, const uint32_t* __restrict__ row_off, uint32_t R, int validate,
                        unsigned long long* __restrict__ flag_counts, unsigned long long* __restrict__ sval,
                        uint8_t* __restrict__ shas, DecMeta* __restrict__ meta) {
  extern __shared__ __align__(16) uint8_t dsm[];
  int32_t* last_row = reinterpret_cast<int32_t*>(dsm);
  const uint32_t* planes = P.planes;
  for (uint32_t u = threadIdx.x; u < P.U; u += DEC_THREADS) last_row[u] = -1;
  __syncthreads();
  const uint32_t r0 = blockIdx.x * R, r1 = min(P.nrows, r0 + R);
  // a row per group of GL lanes: DEC_WARPS * 32 / GL rows are walked at a time
  constexpr uint32_t GPW = 32 / GL;
  const uint32_t first = r0 + (threadIdx.x >> 5) * GPW + lane_id() / GL;
  const uint8_t* rows = P.blk + P.rows_base;
  for (uint32_t r = first; r < r1; r += DEC_WARPS * GPW) {
    const int32_t rl = (int32_t)(r - r0);
    const uint8_t* rp = rows + row_off[r];
    warp_parse_row<GL>(P, planes, rp, first_flag_byte<GL>(P, rp), [&](uint32_t u, uint32_t voff) {
      atomicMax(&last_row[u], rl);
      if (flag_counts) atomicAdd(&flag_counts[u], 1ull);
      if (validate && is_text_like(P.utype[u])) {
        const unsigned long long v = load_le(rp + voff, P.usz[u]);
        if (v != 0 && (uint64_t)(uint32_t)(v + P.ubase[u]) > P.dict_total) meta->err = 1;
      }
    });
  }
  __syncthreads();
  for (uint32_t r = first; r < r1; r += DEC_WARPS * GPW) {
    const int32_t rl = (int32_t)(r - r0);
    const uint8_t* rp = rows + row_off[r];
    warp_parse_row<GL>(P, planes, rp, first_flag_byte<GL>(P, rp), [&](uint32_t u, uint32_t voff) {
      if (last_row[u] == rl) sval[(size_t)blockIdx.x * P.U + u] = load_le(rp + voff, P.usz[u]);
    });
  }
  for (uint32_t u = threadIdx.x; u < P.U; u += DEC_THREADS) shas[(size_t)blockIdx.x * P.U + u] = last_row[u] >= 0 ? 1 : 0;
}

// ---------------------------------------------------------------------------------------------
// formatting
// ---------------------------------------------------------------------------------------------
// An output row is a fixed template - separators, the defaults of unused columns, the terminator - with the text of
// the used columns ("items", in output order) spliced in.  Static segment i precedes item i; segment n_items closes
// the row.  Static byte k of the template therefore lands at k + (dynamic bytes of the items before its segment).
struct FmtTables {
  uint32_t n_items;             // dynamic items (used columns that are output), in output order
  const uint32_t* item_u;       // [n_items] used-column index
  const uint32_t* item_pos;     // [n_items] static bytes in front of the text of item i
  const uint4* sgrp;            // [n_groups] template bytes in groups of 1..4 that never straddle a segment:
                                //   .x = the bytes, .y = segment, .z = offset of the first byte in the template, .w = count
  uint32_t n_groups;
  uint32_t static_total;
  unsigned long long first_row;  // number of the block's first row, for the virtual row-number item
  uint32_t rownum_item;          // index of that item, ITEM_ROWNUM (= none) otherwise
};
constexpr uint32_t ITEM_ROWNUM = 0xffffffffu;  // item_u marker: the item is the running row number, not a used column

// bit i of nulmap = dictionary byte i is NUL; 16 bytes per thread
__global__ void k_dict_nulmap(const uint8_t* __restrict__ dict, uint64_t dict_total, uint32_t* __restrict__ nulmap, uint64_t nwords) {
  const uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= nwords) return;
  uint32_t m = 0;
  const uint64_t b0 = w * 32;
  if (b0 + 36 <= dict_total) {
    const uintptr_t a = reinterpret_cast<uintptr_t>(dict + b0);
    const uint32_t* p = reinterpret_cast<const uint32_t*>(a & ~(uintptr_t)3);
    const uint32_t sh = (uint32_t)(a & 3u) * 8u;
    uint32_t prev = __ldg(p);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const uint32_t nx = __ldg(p + k + 1);
      const uint32_t x = __funnelshift_r(prev, nx, sh);
      prev = nx;
      // exact zero-byte flags (bit 7 of every zero byte), gathered to 4 bits
      const uint32_t z = ~(((x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | x | 0x7F7F7F7Fu);
      m |= movemask4(z) << (4 * k);
    }
  } else {
    for (uint32_t i = 0; i < 32; ++i) {
      const uint64_t b = b0 + i;
      if (b >= dict_total || __ldg(dict + b) == 0) m |= 1u << i;  // everything past the dictionary terminates
    }
  }
  nulmap[w] = m;
}

// strlen of the dictionary entry at byte `index` (GetWord + strlen, UnconvertFromZDW.cpp:359-371,1380), at most room
__device__ __forceinline__ uint32_t dict_strlen(const DecParams& P, uint32_t index, uint64_t room) {
  const uint32_t* bm = P.nulmap + (index >> 5);
  const uint32_t sh = index & 31u;
  uint32_t w = __ldg(bm) >> sh;
  if (w) return (uint32_t)min((uint64_t)(__ffs(w) - 1), room);
  uint64_t pos = 32u - sh;
  for (;;) {
    if (pos >= room) return (uint32_t)room;
    w = __ldg(++bm);
    if (w) return (uint32_t)min(pos + (uint64_t)(__ffs(w) - 1), room);
    pos += 32;
  }
}

// Length of the text of used column u holding stored value v.  Mirrors the switch in readNextRow
// (UnconvertFromZDW.cpp:1349-1453).
__device__ __forceinline__ uint32_t value_len(const DecParams& P, uint32_t u, uint8_t t, unsigned long long v, DecMeta* meta) {
  if (is_text_like(t)) {
    if (v == 0) return t == ZDWB_DECIMAL ? 14u : 0u;  // outputDefault(DECIMAL) = "0.000000000000"
    const uint32_t index = (uint32_t)(v + P.ubase[u]);  // ULONG index: :1363
    if ((uint64_t)index > P.dict_total) {                // :1364 (the reference allows index == dictionarySize)
      meta->err = 1;
      return 0;
    }
    return dict_strlen(P, index, P.dict_total - index);
  }
  if (t == ZDWB_CHAR) {  // :1396-1420
    if (v == 0) return 0;
    const uint8_t b0 = (uint8_t)(v + P.ubase[u]);
    return b0 == (uint8_t)'\\' ? 2u : (b0 ? 1u : 0u);
  }
  const unsigned long long full = v ? v + P.ubase[u] : 0ull;
  if (is_signed_int_type(t) && (long long)full < 0) {
    // lltoa (:333-356): '-' then one character per division step of the negated value (INT64_MIN stays negative
    // and still takes 19 steps)
    const unsigned long long mag = 0ull - full;
    return 1u + digits_u64(mag);
  }
  return digits_u64(full);
}

// The lanes of a row group write the template bytes of a row, one piece of up to 4 bytes of one segment per lane and
// step; the descriptors of four steps are fetched before any of them is used.
template <int G>
__device__ __forceinline__ void warp_write_template(const FmtTables& FT, const uint32_t* __restrict__ ioffj,
                                                    uint8_t* __restrict__ row) {
  for (uint32_t g0 = lane_id() & (unsigned)(G - 1); g0 < FT.n_groups; g0 += 4 * G) {
    uint4 sg[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const uint32_t g = g0 + (uint32_t)(G * k);
      sg[k] = g < FT.n_groups ? __ldg(FT.sgrp + g) : make_uint4(0u, 0u, 0u, 0u);
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if (sg[k].w == 0u) continue;
      uint8_t* d = row + sg[k].z + ioffj[sg[k].y];
      d[0] = (uint8_t)sg[k].x;
      if (sg[k].w > 1) d[1] = (uint8_t)(sg[k].x >> 8);
      if (sg[k].w > 2) d[2] = (uint8_t)(sg[k].x >> 16);
      if (sg[k].w > 3) d[3] = (uint8_t)(sg[k].x >> 24);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// streaming row writer: one warp owns a strip of consecutive rows and walks them in order, keeping for every output
// item (a used column that is output, or the running row number) its text length and, for rendered texts - dictionary
// strings of up to 16 bytes and all numbers - the text itself in shared memory.  A row only touches the items its flag
// bits name; everything else is copied from the warp's state.  No CTA-wide barrier, no cross-warp dependency:
// k_dec_row_lens measures every row first (same walk, lengths only), an exclusive scan turns the lengths into row
// offsets, k_dec_write_rows then assembles each row straight in global memory.
// ---------------------------------------------------------------------------------------------
struct WarpLayout {        // byte offsets inside a warp's slice of dynamic shared memory
  uint32_t o_len, o_val, o_textc, o_ioff, o_llist;
  uint32_t stride;         // bytes per warp
  uint32_t warps;          // warps per CTA
};

constexpr uint32_t LEN_LONG_TEXT = 0x80000000u;  // flag in len[]: the text lives in the dictionary (more than 16 bytes)
constexpr uint32_t LEN_MASK = 0x7fffffffu;

struct WarpState {            // all indexed by output item
  uint32_t* len;              // [NI] text length (| LEN_LONG_TEXT)
  uint32_t* aux;              // [NI] dictionary index of a long text; characters 17..20 of a number
  uint32_t* textc;            // [NI][4] rendered text, first 16 bytes
  uint32_t* ioff;             // [NI + 1]
  uint32_t* llist;            // [1 + NI]  ([0] = count)
};

// New value v for used column u = output item i: updates len[i] and, when WRITE, what the row writer needs to emit it.
template <bool WRITE>
__device__ __forceinline__ void set_column(const DecParams& P, const WarpState& S, uint32_t u, uint32_t i, unsigned long long v,
                                           DecMeta* meta) {
  const uint8_t t = P.utype[u];
  if (is_text_like(t)) {
    if (v == 0) {
      if (t == ZDWB_DECIMAL) {  // outputDefault(DECIMAL): "0.000000000000"
        S.len[i] = 14;
        if (WRITE) {
          uint32_t* tc = S.textc + 4 * (size_t)i;
          tc[0] = 0x30302e30u;
          tc[1] = 0x30303030u;
          tc[2] = 0x30303030u;
          tc[3] = 0x00003030u;
        }
      } else {
        S.len[i] = 0;
      }
      return;
    }
    const uint32_t index = (uint32_t)(v + P.ubase[u]);  // ULONG index: UnconvertFromZDW.cpp:1363
    if ((uint64_t)index > P.dict_total) {                // :1364 (the reference allows index == dictionarySize)
      meta->err = 1;
      S.len[i] = 0;
      return;
    }
    const uint32_t l = dict_strlen(P, index, P.dict_total - index);
    if (l >= LEN_LONG_TEXT) meta->err = 1;  // (cannot happen: a dictionary is smaller than 4 GiB and entries end at a NUL)
    S.len[i] = l > 16 ? (l | LEN_LONG_TEXT) : l;
    if (WRITE) {
      if (l > 16) {
        S.aux[i] = index;  // copied from the dictionary row by row
      } else if (l) {      // short texts are kept rendered
        const uint8_t* s = P.blk + P.dict_base + index;
        const uintptr_t a = reinterpret_cast<uintptr_t>(s);
        const uint32_t* w = reinterpret_cast<const uint32_t*>(a & ~(uintptr_t)3);
        const uint32_t* wend = reinterpret_cast<const uint32_t*>(reinterpret_cast<uintptr_t>(P.blk + P.avail - 1) & ~(uintptr_t)3);
        const uint32_t sh = (uint32_t)(a & 3u) * 8u;
        const uint32_t lim = (uint32_t)min((ptrdiff_t)4, wend - w);
        const uint32_t w0 = __ldg(w), w1 = __ldg(w + min(1u, lim)), w2 = __ldg(w + min(2u, lim)), w3 = __ldg(w + min(3u, lim)),
                       w4 = __ldg(w + min(4u, lim));
        uint32_t* tc = S.textc + 4 * (size_t)i;
        tc[0] = __funnelshift_r(w0, w1, sh);
        tc[1] = __funnelshift_r(w1, w2, sh);
        tc[2] = __funnelshift_r(w2, w3, sh);
        tc[3] = __funnelshift_r(w3, w4, sh);
      }
    }
    return;
  }
  const uint32_t l = value_len(P, u, t, v, meta);
  S.len[i] = l;
  if (WRITE && l) {
    uint32_t* tc = S.textc + 4 * (size_t)i;
    if (t == ZDWB_CHAR) {  // one byte, or a backslash and the byte after it (UnconvertFromZDW.cpp:1396-1420)
      tc[0] = (uint32_t)(v + P.ubase[u]) & 0xffffu;
    } else {  // integers: up to 20 characters, the last four live in the item's aux word
      const unsigned long long full = v ? v + P.ubase[u] : 0ull;
      uint32_t w[5];
      render_int(full, is_signed_int_type(t) && (long long)full < 0, l, w);
      tc[0] = w[0];
      tc[1] = w[1];
      tc[2] = w[2];
      tc[3] = w[3];
      S.aux[i] = w[4];
    }
  }
}

// n bytes from the dictionary to a row by the 8 lanes of an octet: the destination's head up to its next 4-byte boundary
// and its tail go byte by byte (lane 0 / lane 1), everything between as aligned words, one per lane and step, each put
// together from two aligned source words
__device__ __forceinline__ void octet_copy(uint8_t* __restrict__ d, const uint8_t* __restrict__ s, uint32_t n, unsigned gl) {
  const uint32_t head = min(n, (4u - (uint32_t)(reinterpret_cast<uintptr_t>(d) & 3u)) & 3u);
  if (gl == 0) {
    for (uint32_t k = 0; k < head; ++k) d[k] = __ldg(s + k);
  }
  const uint32_t nw = (n - head) >> 2, tail = (n - head) & 3u;
  const uintptr_t a = reinterpret_cast<uintptr_t>(s + head);
  const uint32_t* w = reinterpret_cast<const uint32_t*>(a & ~(uintptr_t)3);
  const uint32_t sh = (uint32_t)(a & 3u) * 8u;
  uint32_t* dw = reinterpret_cast<uint32_t*>(d + head);
  for (uint32_t k = gl; k < nw; k += 8) {
    const uint32_t lo = __ldg(w + k);
    const uint32_t hi = sh ? __ldg(w + k + 1) : 0u;
    dw[k] = __funnelshift_r(lo, hi, sh);
  }
  if (gl == 1) {
    for (uint32_t k = 0; k < tail; ++k) d[head + 4u * nw + k] = __ldg(s + head + 4u * nw + k);
  }
}

__device__ __forceinline__ WarpState warp_state(uint8_t* dsm, const WarpLayout& L, unsigned warp) {
  uint8_t* base = dsm + (size_t)warp * L.stride;
  WarpState S;
  S.len = reinterpret_cast<uint32_t*>(base + L.o_len);
  S.aux = reinterpret_cast<uint32_t*>(base + L.o_val);
  S.textc = reinterpret_cast<uint32_t*>(base + L.o_textc);
  S.ioff = reinterpret_cast<uint32_t*>(base + L.o_ioff);
  S.llist = reinterpret_cast<uint32_t*>(base + L.o_llist);
  return S;
}

// One group of G lanes per strip of RS rows.  WRITE = false: lengths only -> row_len[r].  WRITE = true: rows -> out.
// G = 32 for wide schemas; with at most 8 (16) output items and flag bytes a warp walks 4 (2) strips side by side, so
// that narrow tables do not leave three quarters of every warp idle.
// A cached text goes out as head bytes up to the next 4-byte boundary of the destination, aligned words funnel-shifted
// out of the cache, then tail bytes (measured on C4: 0.90 ms per block against 0.98 with byte-by-byte stores).
template <bool WRITE, int G>
__global__ void __launch_bounds__(128, 10)
    k_dec_rows(const DecParams P, const FmtTables FT, const int32_t* __restrict__ u_item, const uint32_t* __restrict__ row_off,
               uint32_t RS, const WarpLayout L, const unsigned long long* __restrict__ cin, unsigned long long* __restrict__ row_len,
               const unsigned long long* __restrict__ out_row_off, uint8_t* __restrict__ out, DecMeta* __restrict__ meta) {
  extern __shared__ __align__(16) uint8_t dsm[];
  constexpr uint32_t GPW = 32 / G;  // groups per warp
  const unsigned lane = lane_id(), warp = threadIdx.x >> 5;
  const unsigned gl = lane & (unsigned)(G - 1), gm = group_mask<G>();
  const uint32_t group = warp * GPW + lane / G;               // group within the CTA
  const uint32_t strip = blockIdx.x * L.warps * GPW + group;
  const uint32_t r0 = strip * RS;
  if (warp >= L.warps || r0 >= P.nrows) return;
  const uint32_t r1 = min(P.nrows, r0 + RS);
  const WarpState S = warp_state(dsm, L, group);
  const uint32_t U = P.U, NI = FT.n_items;
  const uint8_t* rows = P.blk + P.rows_base;
  const bool has_rownum = FT.rownum_item != ITEM_ROWNUM;

  // ---- state at the start of the strip: the values carried in
  for (uint32_t i = gl; i < NI; i += G) S.len[i] = 0;
  if (gl == 0) S.llist[0] = 0;
  __syncwarp(gm);
  for (uint32_t u = gl; u < U; u += G) {
    const int32_t i = __ldg(u_item + u);
    if (i < 0) continue;  // not output: never touched
    set_column<WRITE>(P, S, u, (uint32_t)i, cin[(size_t)strip * U + u], meta);
  }
  __syncwarp(gm);
  long long dyn = 0;  // dynamic bytes of the current row without the row number (lane-local share; summed when needed)
  for (uint32_t i = gl; i < NI; i += G) dyn += S.len[i] & LEN_MASK;

  // the row's offset and its first flag bytes are fetched one row ahead
  uint32_t ro = row_off[r0];
  uint32_t fb = first_flag_byte<G>(P, rows + ro);
  for (uint32_t r = r0; r < r1; ++r) {
    const uint8_t* rp = rows + ro;
    const uint32_t fb_now = fb;
    if (r + 1 < r1) {
      ro = row_off[r + 1];
      fb = first_flag_byte<G>(P, rows + ro);
    }
    // ---- the columns this row changes: the flag walk only lists them, the values are then applied G at a time
    warp_parse_row<G>(P, P.planes, rp, fb_now, [&](uint32_t u, uint32_t voff) {
      if (__ldg(u_item + u) < 0) return;
      const uint32_t e = atomicAdd(&S.llist[0], 1u);
      S.llist[1 + e] = u;
      S.ioff[e] = voff;
    });
    __syncwarp(gm);
    {
      const uint32_t n = S.llist[0];
      int32_t delta = 0;
      for (uint32_t e = gl; e < n; e += G) {
        const uint32_t u = S.llist[1 + e];
        const uint32_t i = (uint32_t)__ldg(u_item + u);
        const unsigned long long v = load_le(rp + S.ioff[e], P.usz[u]);
        const int32_t old = (int32_t)(S.len[i] & LEN_MASK);
        set_column<WRITE>(P, S, u, i, v, meta);
        delta += (int32_t)(S.len[i] & LEN_MASK) - old;
      }
      dyn += delta;
      if (WRITE && has_rownum && gl == 0) {  // virtual_export_row (UnconvertFromZDW.cpp:1256-1261): a number like any other
        const unsigned long long x = FT.first_row + r;
        const uint32_t l = digits_u64(x);
        uint32_t w[5];
        render_int(x, false, l, w);
        uint32_t* tc = S.textc + 4 * (size_t)FT.rownum_item;
        tc[0] = w[0];
        tc[1] = w[1];
        tc[2] = w[2];
        tc[3] = w[3];
        S.aux[FT.rownum_item] = w[4];
        S.len[FT.rownum_item] = l;
      }
      __syncwarp(gm);
      if (gl == 0) S.llist[0] = 0;
      __syncwarp(gm);
    }

    if (!WRITE) {
      long long tot = dyn;
#pragma unroll
      for (int o = G / 2; o > 0; o >>= 1) tot += __shfl_xor_sync(gm, tot, o, G);
      if (gl == 0) {
        unsigned long long rl = (unsigned long long)tot + FT.static_total;
        if (has_rownum) rl += digits_u64(FT.first_row + r);
        row_len[r] = rl;
      }
      continue;
    }

    // ---- offset of every item's text among the dynamic bytes of the row
    uint32_t run = 0;
    for (uint32_t i0 = 0; i0 < NI; i0 += G) {
      const uint32_t i = i0 + gl;
      const uint32_t l = i < NI ? (S.len[i] & LEN_MASK) : 0u;
      uint32_t inc = l;
#pragma unroll
      for (int o = 1; o < G; o <<= 1) {
        uint32_t t = __shfl_up_sync(gm, inc, o, G);
        if (gl >= (unsigned)o) inc += t;
      }
      if (i < NI) S.ioff[i] = run + inc - l;
      run += __shfl_sync(gm, inc, G - 1, G);
    }
    if (gl == 0) S.ioff[NI] = run;
    __syncwarp(gm);
    uint8_t* dst = out + out_row_off[r];

    // ---- template, then the items
    warp_write_template<G>(FT, S.ioff, dst);
    for (uint32_t i0 = 0; i0 < NI; i0 += G) {
      const uint32_t i = i0 + gl;
      if (i >= NI) continue;
      const uint32_t lf = S.len[i], l = lf & LEN_MASK;
      if (!l) continue;
      if (lf & LEN_LONG_TEXT) {
        S.llist[1 + atomicAdd(&S.llist[0], 1u)] = i;
        continue;
      }
      // rendered text: 16 bytes in the cache, numbers up to 4 more in aux
      uint8_t* d = dst + __ldg(FT.item_pos + i) + S.ioff[i];
      const uint32_t* tw = S.textc + 4 * (size_t)i;
      const uint32_t x4 = S.aux[i];  // characters 17..20 of a number (not read as text for anything shorter)
      auto X = [&](uint32_t j) { return j < 4u ? tw[j] : x4; };
      const uint32_t head = min(l, (4u - (uint32_t)(reinterpret_cast<uintptr_t>(d) & 3u)) & 3u);
      const uint32_t x0 = tw[0];
      if (head > 0) d[0] = (uint8_t)x0;
      if (head > 1) d[1] = (uint8_t)(x0 >> 8);
      if (head > 2) d[2] = (uint8_t)(x0 >> 16);
      const uint32_t rest = l - head, nw = rest >> 2, sh = head * 8u;
      uint32_t* dw = reinterpret_cast<uint32_t*>(d + head);  // 4-byte aligned by construction
      for (uint32_t m = 0; m < nw; ++m) dw[m] = __funnelshift_r(X(m), X(min(m + 1u, 4u)), sh);
      const uint32_t tail = rest & 3u;
      if (tail) {
        const uint32_t t = __funnelshift_r(X(nw), X(min(nw + 1u, 4u)), sh);
        uint8_t* dt = d + head + 4u * nw;
        dt[0] = (uint8_t)t;
        if (tail > 1) dt[1] = (uint8_t)(t >> 8);
        if (tail > 2) dt[2] = (uint8_t)(t >> 16);
      }
    }
    __syncwarp(gm);
    {
      const uint32_t n = S.llist[0];
      for (uint32_t e = gl >> 3; e < n; e += G / 8) {  // the octets of the group
        const uint32_t i = S.llist[1 + e];
        octet_copy(dst + __ldg(FT.item_pos + i) + S.ioff[i], P.blk + P.dict_base + S.aux[i], S.len[i] & LEN_MASK, gl & 7u);
      }
      __syncwarp(gm);
      if (gl == 0) S.llist[0] = 0;
    }
    __syncwarp(gm);
  }
}

// ---------------------------------------------------------------------------------------------
// delta row writer (wide schemas): a decoded row differs from the row before only in the items whose flag bit is set -
// 16 % of the cells of analytics-shaped data - and everything between two changed items, separators and defaults
// included, is a byte-for-byte copy of the same stretch of the previous row, moved by the length changes so far.
// The previous row has just been written by the same warp (it sits in L2), so row r is assembled from it: 16-byte
// chunks whose bytes all come from one unchanged stretch are copied with one unaligned load and one aligned store,
// only the changed items are rendered (readNextRow's per-column switch, UnconvertFromZDW.cpp:1349-1453), and the few
// chunks that straddle a changed item go byte by byte.  The first row of a strip - and a row with more changes than
// the warp's lists hold - is assembled in full from the column values the warp keeps.
// ---------------------------------------------------------------------------------------------
constexpr uint32_t DLC = 64;   // changed items per row the delta path handles (more: the row is assembled in full)

struct DeltaLayout {   // byte offsets inside a warp's slice of dynamic shared memory
  uint32_t o_val, o_len, o_ioff, o_lcs, o_lce, o_lpe, o_lvoff, o_litem, o_lu, o_slow;
  uint32_t stride, warps;
};
struct DeltaState {
  unsigned long long* val;  // [NI] stored value of the item's column
  uint32_t* len;            // [NI] length of its text
  uint32_t* ioff;           // [NI + 1] dynamic bytes in front of the item (prefix of len)
  uint32_t *lcs, *lce, *lpe;  // [DLC] changed item: start / end in this row, end in the previous row
  uint32_t* lvoff;          // [DLC] offset of its value in the encoded row
  uint16_t *litem, *lu;     // [DLC] its item / used column
  uint16_t* slow;           // [max(2 DLC + 4, NI)] chunks that straddle a changed item or the row's ends; afterwards (lng)
  uint16_t* lng;            // the items whose text comes straight from the dictionary, by octets (same memory)
};
__device__ __forceinline__ DeltaState delta_state(uint8_t* dsm, const DeltaLayout& L, unsigned warp) {
  uint8_t* b = dsm + (size_t)warp * L.stride;
  DeltaState S;
  S.val = reinterpret_cast<unsigned long long*>(b + L.o_val);
  S.len = reinterpret_cast<uint32_t*>(b + L.o_len);
  S.ioff = reinterpret_cast<uint32_t*>(b + L.o_ioff);
  S.lcs = reinterpret_cast<uint32_t*>(b + L.o_lcs);
  S.lce = reinterpret_cast<uint32_t*>(b + L.o_lce);
  S.lpe = reinterpret_cast<uint32_t*>(b + L.o_lpe);
  S.lvoff = reinterpret_cast<uint32_t*>(b + L.o_lvoff);
  S.litem = reinterpret_cast<uint16_t*>(b + L.o_litem);
  S.lu = reinterpret_cast<uint16_t*>(b + L.o_lu);
  S.slow = reinterpret_cast<uint16_t*>(b + L.o_slow);
  S.lng = S.slow;
  return S;
}

__device__ __forceinline__ uint32_t ld_coherent_u32(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// 16 bytes from an arbitrary address (coherent loads: five aligned words, funnel shifts)
__device__ __forceinline__ uint4 ld_coherent_16(const uint8_t* s) {
  const uintptr_t a = reinterpret_cast<uintptr_t>(s);
  const uint32_t* w = reinterpret_cast<const uint32_t*>(a & ~(uintptr_t)3);
  const uint32_t sh = (uint32_t)(a & 3u) * 8u;
  const uint32_t w0 = ld_coherent_u32(w), w1 = ld_coherent_u32(w + 1), w2 = ld_coherent_u32(w + 2), w3 = ld_coherent_u32(w + 3),
                 w4 = sh ? ld_coherent_u32(w + 4) : 0u;
  uint4 v;
  v.x = __funnelshift_r(w0, w1, sh);
  v.y = __funnelshift_r(w1, w2, sh);
  v.z = __funnelshift_r(w2, w3, sh);
  v.w = __funnelshift_r(w3, w4, sh);
  return v;
}
// word `at` .. `at` + 3 of a 16-byte chunk: the bytes [from, upto) of the chunk are taken from v, the others stay
__device__ __forceinline__ uint32_t merge_bytes(uint32_t acc, uint32_t v, uint32_t from, uint32_t upto, uint32_t at) {
  const uint32_t lo = from > at ? min(from - at, 4u) : 0u, hi = upto > at ? min(upto - at, 4u) : 0u;  // bytes [lo, hi) of the word
  if (hi <= lo) return acc;
  const uint32_t m = (hi >= 4u ? 0xffffffffu : ((1u << (8u * hi)) - 1u)) & ~((1u << (8u * lo)) - 1u);
  return (acc & ~m) | (v & m);
}

// l (1..20) bytes held in w[0..4] (first byte = lowest byte of w[0]) to d: head bytes up to the next 4-byte boundary,
// aligned words, tail bytes
__device__ __forceinline__ void emit_words(uint8_t* __restrict__ d, const uint32_t w[5], uint32_t l) {
  const uint32_t head = min(l, (4u - (uint32_t)(reinterpret_cast<uintptr_t>(d) & 3u)) & 3u);
  if (head > 0) d[0] = (uint8_t)w[0];
  if (head > 1) d[1] = (uint8_t)(w[0] >> 8);
  if (head > 2) d[2] = (uint8_t)(w[0] >> 16);
  const uint32_t rest = l - head, nw = rest >> 2, sh = head * 8u;
  uint32_t* dw = reinterpret_cast<uint32_t*>(d + head);
  if (nw > 0) dw[0] = __funnelshift_r(w[0], w[1], sh);
  if (nw > 1) dw[1] = __funnelshift_r(w[1], w[2], sh);
  if (nw > 2) dw[2] = __funnelshift_r(w[2], w[3], sh);
  if (nw > 3) dw[3] = __funnelshift_r(w[3], w[4], sh);
  if (nw > 4) dw[4] = w[4] >> sh;
  const uint32_t tail = rest & 3u;
  if (tail) {
    const uint32_t lo = nw == 0 ? w[0] : nw == 1 ? w[1] : nw == 2 ? w[2] : nw == 3 ? w[3] : w[4];
    const uint32_t hi = nw == 0 ? w[1] : nw == 1 ? w[2] : nw == 2 ? w[3] : nw == 3 ? w[4] : 0u;
    const uint32_t t = __funnelshift_r(lo, hi, sh);
    uint8_t* dt = d + head + 4u * nw;
    dt[0] = (uint8_t)t;
    if (tail > 1) dt[1] = (uint8_t)(t >> 8);
    if (tail > 2) dt[2] = (uint8_t)(t >> 16);
  }
}

// Text of used column u holding stored value v (l = its length, > 0) to d.  Returns false for a dictionary text of
// more than 16 bytes: the caller copies those with the octets of the warp.
__device__ __forceinline__ bool emit_value(const DecParams& P, uint32_t u, unsigned long long v, uint32_t l, uint8_t* __restrict__ d) {
  const uint8_t t = P.utype[u];
  uint32_t w[5] = {0u, 0u, 0u, 0u, 0u};
  if (is_text_like(t)) {
    if (v == 0) {  // outputDefault(DECIMAL): "0.000000000000"
      w[0] = 0x30302e30u;
      w[1] = 0x30303030u;
      w[2] = 0x30303030u;
      w[3] = 0x00003030u;
    } else {
      if (l > 16) return false;
      const uint32_t index = (uint32_t)(v + P.ubase[u]);
      const uint8_t* s = P.blk + P.dict_base + index;
      const uintptr_t a = reinterpret_cast<uintptr_t>(s);
      const uint32_t* p = reinterpret_cast<const uint32_t*>(a & ~(uintptr_t)3);
      const uint32_t* pend = reinterpret_cast<const uint32_t*>(reinterpret_cast<uintptr_t>(P.blk + P.avail - 1) & ~(uintptr_t)3);
      const uint32_t sh = (uint32_t)(a & 3u) * 8u;
      const uint32_t lim = (uint32_t)min((ptrdiff_t)4, pend - p);
      const uint32_t w0 = __ldg(p), w1 = __ldg(p + min(1u, lim)), w2 = __ldg(p + min(2u, lim)), w3 = __ldg(p + min(3u, lim)),
                     w4 = __ldg(p + min(4u, lim));
      w[0] = __funnelshift_r(w0, w1, sh);
      w[1] = __funnelshift_r(w1, w2, sh);
      w[2] = __funnelshift_r(w2, w3, sh);
      w[3] = __funnelshift_r(w3, w4, sh);
    }
  } else if (t == ZDWB_CHAR) {
    w[0] = (uint32_t)(v + P.ubase[u]) & 0xffffu;
  } else {
    const unsigned long long full = v ? v + P.ubase[u] : 0ull;
    render_int(full, is_signed_int_type(t) && (long long)full < 0, l, w);
  }
  emit_words(d, w, l);
  return true;
}

// exclusive prefix of S.len over the items -> S.ioff (all lanes)
__device__ __forceinline__ void delta_scan_lens(const DeltaState& S, uint32_t NI) {
  const unsigned lane = lane_id();
  uint32_t run = 0;
  for (uint32_t i0 = 0; i0 < NI; i0 += 32) {
    const uint32_t i = i0 + lane;
    const uint32_t l = i < NI ? S.len[i] : 0u;
    uint32_t inc = l;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= (unsigned)o) inc += t;
    }
    if (i < NI) S.ioff[i] = run + inc - l;
    run += __shfl_sync(0xffffffffu, inc, 31);
  }
  if (lane == 0) S.ioff[NI] = run;
}

__global__ void __launch_bounds__(128, 8)
    k_dec_write_delta(const DecParams P, const FmtTables FT, const int32_t* __restrict__ u_item, const uint8_t* __restrict__ outmask,
                      const uint32_t* __restrict__ row_off, uint32_t RS, const DeltaLayout L, const unsigned long long* __restrict__ cin,
                      const unsigned long long* __restrict__ out_row_off, uint8_t* __restrict__ out, DecMeta* __restrict__ meta) {
  extern __shared__ __align__(16) uint8_t dsm[];
  const unsigned lane = lane_id(), warp = threadIdx.x >> 5;
  const uint32_t strip = blockIdx.x * L.warps + warp;
  const uint32_t r0 = strip * RS;
  if (warp >= L.warps || r0 >= P.nrows) return;
  const uint32_t r1 = min(P.nrows, r0 + RS);
  const DeltaState S = delta_state(dsm, L, warp);
  const uint32_t U = P.U, NI = FT.n_items, F = P.F;
  const uint8_t* rows = P.blk + P.rows_base;

  // ---- the values carried into the strip
  for (uint32_t u = lane; u < U; u += 32) {
    const int32_t i = __ldg(u_item + u);
    if (i < 0) continue;
    const unsigned long long v = cin[(size_t)strip * U + u];
    S.val[i] = v;
    S.len[i] = value_len(P, u, P.utype[u], v, meta);
  }
  __syncwarp();
  const uint8_t* prev = nullptr;  // the previous row of the strip in `out`
  const unsigned long long strip_end = out_row_off[r1], strip_begin = out_row_off[r0];

  for (uint32_t r = r0; r < r1; ++r) {
    const uint8_t* rp = rows + row_off[r];
    const unsigned long long o0 = out_row_off[r];
    uint8_t* dst = out + o0;
    const uint32_t row_len = (uint32_t)(out_row_off[r + 1] - o0);
    // ---- which items change?  flag byte j: bits of the used columns 8 j .. 8 j + 7; the value bytes in front of a
    // flag byte's values come from the width bit planes like in warp_parse_row
    uint32_t n = 0;         // changed items that are output
    bool full = prev == nullptr;
    if (!full) {            // more changes than the lists hold?  (then the values are applied on the spot, see below)
      uint32_t cnt = 0;
      for (uint32_t j = lane; j < F; j += 32) cnt += (uint32_t)__popc((uint32_t)__ldg(rp + j) & (uint32_t)__ldg(outmask + j));
      full = __reduce_add_sync(0xffffffffu, cnt) > DLC;
    }
    uint32_t run = F;       // offset of the next value inside the encoded row
    for (uint32_t j0 = 0; j0 < F; j0 += 32) {
      const uint32_t j = j0 + lane;
      uint32_t fb = 0, bl = 0, ob = 0;
      if (j < F) {
        fb = (uint32_t)__ldg(rp + j);
        if (fb) {
          const uint32_t sh = (j & 3u) * 8u, w = j >> 2;
          bl = __popc(fb & (P.planes[w] >> sh)) + 2u * __popc(fb & (P.planes[P.W + w] >> sh)) +
               4u * __popc(fb & (P.planes[2 * P.W + w] >> sh)) + 8u * __popc(fb & (P.planes[3 * P.W + w] >> sh));
          ob = fb & (uint32_t)__ldg(outmask + j);
        }
      }
      const uint32_t mine = bl | ((uint32_t)__popc(ob) << 16);
      uint32_t inc = mine;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= (unsigned)o) inc += t;
      }
      const uint32_t tot = __shfl_sync(0xffffffffu, inc, 31);
      uint32_t voff = run + ((inc - mine) & 0xffffu);
      uint32_t at = n + ((inc - mine) >> 16);
      const uint32_t cnt_all = tot >> 16;
      // every flagged column: the new value (and, on the delta path, its place in the list)
      while (fb) {
        const int b = __ffs(fb) - 1;
        fb &= fb - 1;
        const uint32_t u = j * 8 + b;
        if (u >= U) break;
        const uint32_t sz = P.usz[u];
        if ((ob >> b) & 1u) {
          if (!full) {
            S.lu[at] = (uint16_t)u;
            S.lvoff[at] = voff;
          } else {
            const uint32_t i = (uint32_t)__ldg(u_item + u);
            const unsigned long long v = load_le(rp + voff, sz);
            S.val[i] = v;
            S.len[i] = value_len(P, u, P.utype[u], v, meta);
          }
          ++at;
        }
        voff += sz;
      }
      run += tot & 0xffffu;
      n += cnt_all;
    }
    __syncwarp();
    if (!full) {
      // ---- apply the changes: value, new length; where the item ended in the previous row.  Bit 15 of litem marks a
      // change of LENGTH: only those move the bytes behind them
      for (uint32_t e = lane; e < n; e += 32) {
        const uint32_t u = S.lu[e];
        const uint32_t i = (uint32_t)__ldg(u_item + u);
        const unsigned long long v = load_le(rp + S.lvoff[e], P.usz[u]);
        const uint32_t oldl = S.len[i], newl = value_len(P, u, P.utype[u], v, meta);
        S.lpe[e] = __ldg(FT.item_pos + i) + S.ioff[i] + oldl;
        S.litem[e] = (uint16_t)(i | (oldl != newl ? 0x8000u : 0u));
        S.val[i] = v;
        S.len[i] = newl;
      }
      __syncwarp();
    }
    delta_scan_lens(S, NI);
    __syncwarp();

    if (full) {
      // ---- the whole row from the template and the column values
      warp_write_template<32>(FT, S.ioff, dst);
      uint32_t nlong = 0;
      for (uint32_t i0 = 0; i0 < NI; i0 += 32) {
        const uint32_t i = i0 + lane;
        bool is_long = false;
        if (i < NI) {
          const uint32_t l = S.len[i];
          if (l) is_long = !emit_value(P, __ldg(FT.item_u + i), S.val[i], l, dst + __ldg(FT.item_pos + i) + S.ioff[i]);
        }
        const unsigned m = __ballot_sync(0xffffffffu, is_long);
        if (is_long) S.lng[nlong + __popc(m & lanemask_lt())] = (uint16_t)i;
        nlong += __popc(m);
      }
      __syncwarp();
      for (uint32_t e = lane >> 3; e < nlong; e += 4) {
        const uint32_t i = S.lng[e];
        const uint32_t u = __ldg(FT.item_u + i);
        octet_copy(dst + __ldg(FT.item_pos + i) + S.ioff[i], P.blk + P.dict_base + (uint32_t)(S.val[i] + P.ubase[u]), S.len[i], lane & 7u);
      }
    } else {
      // ---- the items whose length changed, in row order: start / end in this row (lcs / lce) and end in the previous
      // row (lpe, compacted in place).  Stretch k (behind such an item k, k = -1: the row's head) holds the bytes
      // [lce[k], lcs[k + 1]) of this row = the previous row's bytes from lpe[k] on.
      uint32_t nb = 0;
      for (uint32_t e0 = 0; e0 < n; e0 += 32) {
        const uint32_t e = e0 + lane;
        uint32_t li = 0, pe = 0;
        if (e < n) {
          li = S.litem[e];
          pe = S.lpe[e];
        }
        const bool moved = (li & 0x8000u) != 0u;
        const unsigned m = __ballot_sync(0xffffffffu, moved);
        __syncwarp();
        if (moved) {
          const uint32_t i = li & 0x7fffu, k = nb + (uint32_t)__popc(m & lanemask_lt());
          const uint32_t cs = __ldg(FT.item_pos + i) + S.ioff[i];
          S.lcs[k] = cs;
          S.lce[k] = cs + S.len[i];
          S.lpe[k] = pe;
        }
        nb += (uint32_t)__popc(m);
        __syncwarp();
      }
      // ---- 16 aligned bytes per lane.  A chunk inside one stretch is one unaligned load; the others - the row's head
      // (its first bytes belong to the row before), chunks that hold an item whose length changed - are merged from
      // their sources afterwards.  Bytes of changed items are overwritten by the rendering below; a chunk may run over
      // the end of the row into the next row of the strip (which is written later), never into another strip.
      const uint32_t a0 = (uint32_t)(reinterpret_cast<uintptr_t>(dst) & 15u);
      const uint32_t nch = (a0 + row_len + 15u) >> 4;
      // (... of the strip: with rows shorter than a chunk the overrun could otherwise pass the rows behind it)
      const uint32_t ext = (uint32_t)min((unsigned long long)row_len + 16ull, strip_end - o0);
      uint32_t nslow = 0, kb = 0;  // kb: moved items that end in front of the round's first chunk (all lanes agree)
      for (uint32_t c0 = 0; c0 < nch; c0 += 32) {
        const uint32_t c = c0 + lane;
        const int32_t x0 = (int32_t)(c * 16u) - (int32_t)a0;  // row-relative offset of the chunk
        bool slow = false;
        uint32_t lo = kb;  // moved items that end at or in front of x: a round's 512 bytes hold few of them
        if (c < nch) {
          const uint32_t x = x0 > 0 ? (uint32_t)x0 : 0u;
          while (lo < nb && S.lce[lo] <= x) ++lo;
          const uint32_t stop = lo < nb ? S.lcs[lo] : ext;  // the stretch ends here
          if (x0 >= 0 && (uint32_t)x0 + 16u <= stop) {
            const uint32_t src = lo ? (uint32_t)x0 - S.lce[lo - 1] + S.lpe[lo - 1] : (uint32_t)x0;
            *reinterpret_cast<uint4*>(dst + x0) = ld_coherent_16(prev + src);
          } else if (!(x0 >= 0 && lo < nb && S.lcs[lo] <= x && (uint32_t)x0 + 16u <= S.lce[lo])) {
            slow = true;  // (a chunk inside one moved item is left to the rendering: at most two listed chunks per item)
          }
        }
        const unsigned m = __ballot_sync(0xffffffffu, slow);
        if (slow) S.slow[nslow + __popc(m & lanemask_lt())] = (uint16_t)c;
        nslow += __popc(m);
        kb = __shfl_sync(0xffffffffu, lo, 31);  // (lanes beyond the last chunk carry the round's start value: harmless)
      }
      __syncwarp();
      for (uint32_t q = lane; q < nslow; q += 32) {
        const uint32_t c = S.slow[q];
        const int32_t x0 = (int32_t)(c * 16u) - (int32_t)a0;
        uint8_t* at = dst + x0;  // 16-byte aligned
        uint4 acc = x0 < 0 ? ld_coherent_16(at) : make_uint4(0u, 0u, 0u, 0u);  // the bytes in front of the row stay
        uint32_t pos = x0 < 0 ? a0 : 0u;  // bytes of the chunk settled so far
        uint32_t k = 0;
        {
          const uint32_t x = x0 > 0 ? (uint32_t)x0 : 0u;
          uint32_t lo = 0, hi = nb;
          while (lo < hi) {
            const uint32_t m = (lo + hi) >> 1;
            if (S.lce[m] <= x) lo = m + 1;
            else hi = m;
          }
          k = lo;
        }
        // source after source: stretch k - 1 up to the start of moved item k, whose bytes are left to the rendering
        while (pos < 16u) {
          const uint32_t x = (uint32_t)(x0 + (int32_t)pos);
          const uint32_t stop = k < nb ? S.lcs[k] : 0xffffffffu;
          uint32_t upto = 16u;  // bytes [pos, upto) of the chunk come from stretch k - 1
          if (stop != 0xffffffffu && stop < (uint32_t)(x0 + 16)) upto = stop > x ? stop - (uint32_t)x0 : pos;
          if (upto > pos) {
            const uint32_t src = k ? x - S.lce[k - 1] + S.lpe[k - 1] : x;
            const uint4 v = ld_coherent_16(prev + src - pos);  // byte j of v = the chunk's byte j
            acc.x = merge_bytes(acc.x, v.x, pos, upto, 0u);
            acc.y = merge_bytes(acc.y, v.y, pos, upto, 4u);
            acc.z = merge_bytes(acc.z, v.z, pos, upto, 8u);
            acc.w = merge_bytes(acc.w, v.w, pos, upto, 12u);
          }
          if (k >= nb) break;
          // skip moved item k (its bytes are rendered below) and go on behind it
          const uint32_t end = S.lce[k];
          pos = end > (uint32_t)(x0 + 16) ? 16u : (end > x ? end - (uint32_t)x0 : max(pos, upto));
          if (pos < upto) pos = upto;
          ++k;
        }
        // bytes of another strip - in front of this strip's first row, behind its last - belong to another warp, which may
        // be writing them right now: such a chunk is stored byte by byte, this row's bytes only
        if ((uint32_t)(x0 + 16) > ext || (x0 < 0 && o0 - (unsigned long long)(-x0) < strip_begin)) {
          const uint32_t w[4] = {acc.x, acc.y, acc.z, acc.w};
          for (int32_t b = x0 < 0 ? -x0 : 0; b < 16 && (uint32_t)(x0 + b) < row_len; ++b) at[b] = (uint8_t)(w[b >> 2] >> (8 * (b & 3)));
        } else {
          *reinterpret_cast<uint4*>(at) = acc;
        }
      }
      __syncwarp();
      // ---- the changed items
      uint32_t nlong = 0;
      for (uint32_t e0 = 0; e0 < n; e0 += 32) {
        const uint32_t e = e0 + lane;
        bool is_long = false;
        if (e < n) {
          const uint32_t i = S.litem[e] & 0x7fffu, l = S.len[i];
          if (l) is_long = !emit_value(P, S.lu[e], S.val[i], l, dst + __ldg(FT.item_pos + i) + S.ioff[i]);
        }
        const unsigned m = __ballot_sync(0xffffffffu, is_long);
        if (is_long) S.lng[nlong + __popc(m & lanemask_lt())] = (uint16_t)e;
        nlong += __popc(m);
      }
      __syncwarp();
      for (uint32_t q = lane >> 3; q < nlong; q += 4) {
        const uint32_t e = S.lng[q];
        const uint32_t i = S.litem[e] & 0x7fffu, u = S.lu[e];
        octet_copy(dst + __ldg(FT.item_pos + i) + S.ioff[i], P.blk + P.dict_base + (uint32_t)(S.val[i] + P.ubase[u]), S.len[i], lane & 7u);
      }
    }
    __syncwarp();
    prev = dst;
  }
}

// ---------------------------------------------------------------------------------------------
// columnar decode (zdwb_decode_columns): the value every selected column holds in every row, as one int64 per cell.
// Text-like columns become dictionary codes: the rank of the entry among the block's dictionary entries, which are
// sorted, so codes compare like the strings.
// ---------------------------------------------------------------------------------------------
// An entry starts at byte p in [1, dict_total) iff byte p - 1 is NUL.  The NULs that start an entry are those at
// q < dict_total - 1: word w of the NUL map with the others cleared.
__device__ __forceinline__ uint32_t entry_nuls(const uint32_t* __restrict__ nulmap, uint64_t dict_total, uint64_t w) {
  const uint64_t lim = dict_total ? dict_total - 1 : 0, b0 = w * 32;
  if (b0 >= lim) return 0u;
  const uint32_t m = __ldg(nulmap + w);
  return lim - b0 >= 32 ? m : m & ((1u << (uint32_t)(lim - b0)) - 1u);
}

// cnt[w] = entries whose NUL lies in word w of the NUL map
__global__ void k_dict_counts(const uint32_t* __restrict__ nulmap, uint64_t dict_total, uint32_t* __restrict__ cnt, uint64_t nwords) {
  const uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (w < nwords) cnt[w] = __popc(entry_nuls(nulmap, dict_total, w));
}

// entry_off[e] = first byte of entry e (prefix = exclusive prefix of cnt); the word of the last NUL map word also writes
// entry_off[entries] = dict_total
__global__ void k_dict_entries(const uint32_t* __restrict__ nulmap, uint64_t dict_total, const uint32_t* __restrict__ prefix,
                               uint64_t nwords, unsigned long long* __restrict__ entry_off) {
  const uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= nwords) return;
  uint32_t m = entry_nuls(nulmap, dict_total, w);
  uint32_t e = prefix[w];
  while (m) {
    const uint32_t b = (uint32_t)__ffs(m) - 1u;
    m &= m - 1u;
    entry_off[e++] = w * 32 + b + 1;
  }
  if (w == nwords - 1) entry_off[e] = dict_total;
}

__device__ __forceinline__ uint32_t low_bits(uint32_t b) { return (1u << b) - 1u; }  // b < 32

// flag word w of a row (flag bytes 4w .. 4w+3; bytes past the F flag bytes read as 0)
__device__ __forceinline__ uint32_t row_flag_word(const DecParams& P, const uint8_t* __restrict__ rp, uint32_t w) {
  uint32_t x = 0;
#pragma unroll
  for (uint32_t b = 0; b < 4; ++b) {
    const uint32_t j = 4 * w + b;
    if (j < P.F) x |= (uint32_t)__ldg(rp + j) << (8 * b);
  }
  return x;
}

// The int64 of a cell of used column u holding stored value v (include/zdw_b200.h, zdwb_decode_columns).  A text offset
// that is not the start of a dictionary entry sets meta->err.
__device__ __forceinline__ unsigned long long column_cell(const DecParams& P, uint32_t u, unsigned long long v,
                                                          const uint32_t* __restrict__ dict_prefix, DecMeta* meta) {
  if (!is_text_like(P.utype[u])) return v ? v + P.ubase[u] : 0ull;
  if (v == 0) return ~0ull;  // -1: no value
  const uint32_t o = (uint32_t)(v + P.ubase[u]);  // ULONG index, UnconvertFromZDW.cpp:1363
  if (o == 0 || (uint64_t)o >= P.dict_total || !((__ldg(P.nulmap + ((o - 1) >> 5)) >> ((o - 1) & 31u)) & 1u)) {
    meta->err = 1;
    return ~0ull;
  }
  return (unsigned long long)(__ldg(dict_prefix + (o >> 5)) + __popc(__ldg(P.nulmap + (o >> 5)) & low_bits(o & 31u)) - 1u);
}

// One warp per strip of 32 rows, one lane per row.  A lane walks the selected used columns in ascending order and keeps
// the offset of the next value in its row from popcounts of its flag bits against the width bit planes.  A row whose
// flag bit is clear takes the value of the nearest lane in front that has one (a ballot and one shuffle), or the
// strip's carry-in.  The warp stores the 32 rows of a column side by side: 256 bytes per column and strip.
__global__ void __launch_bounds__(DEC_THREADS)
    k_dec_columns(const DecParams P, const uint32_t* __restrict__ row_off, const unsigned long long* __restrict__ cin,
                  const uint32_t* __restrict__ sel_u, const uint32_t* __restrict__ sel_k, uint32_t n_sel,
                  const uint32_t* __restrict__ dict_prefix, unsigned long long* __restrict__ values, DecMeta* __restrict__ meta) {
  const unsigned lane = lane_id();
  const uint32_t strip = blockIdx.x * DEC_WARPS + (threadIdx.x >> 5);
  const uint32_t r0 = strip * 32;
  if (r0 >= P.nrows) return;  // (the whole warp)
  const uint32_t r = r0 + lane;
  const bool live = r < P.nrows;
  const uint8_t* rp = P.blk + P.rows_base + (live ? row_off[r] : 0u);
  const unsigned le = lanemask_lt() | (1u << lane);
  uint32_t voff = P.F;  // offset of the next value in the row
  uint32_t cw = 0;      // flag word of the walk, its bits below `from` are counted in voff
  uint32_t from = 0;
  uint32_t fw = live ? row_flag_word(P, rp, 0) : 0u;
  uint32_t pl0 = __ldg(P.planes), pl1 = __ldg(P.planes + P.W), pl2 = __ldg(P.planes + 2 * P.W), pl3 = __ldg(P.planes + 3 * P.W);
  auto widths = [&](uint32_t m) { return __popc(m & pl0) + 2u * __popc(m & pl1) + 4u * __popc(m & pl2) + 8u * __popc(m & pl3); };
  for (uint32_t j = 0; j < n_sel; ++j) {
    const uint32_t u = __ldg(sel_u + j);
    const uint32_t w = u >> 5, b = u & 31u;
    while (cw < w) {
      voff += widths(fw & ~low_bits(from));
      ++cw;
      from = 0;
      fw = live ? row_flag_word(P, rp, cw) : 0u;
      pl0 = __ldg(P.planes + cw);
      pl1 = __ldg(P.planes + P.W + cw);
      pl2 = __ldg(P.planes + 2 * P.W + cw);
      pl3 = __ldg(P.planes + 3 * P.W + cw);
    }
    voff += widths(fw & low_bits(b) & ~low_bits(from));
    from = b;
    const bool has = (fw >> b) & 1u;
    unsigned long long v = has ? load_le(rp + voff, P.usz[u]) : 0ull;
    const unsigned src = __ballot_sync(0xffffffffu, has) & le;
    v = __shfl_sync(0xffffffffu, v, src ? 31 - __clz(src) : lane);
    if (!src) v = cin[(size_t)strip * P.U + u];
    if (live) values[(size_t)__ldg(sel_k + j) * P.nrows + r] = column_cell(P, u, v, dict_prefix, meta);
  }
}

struct HostBlockHeader {
  uint32_t nrows = 0, line_len = 0;
  uint8_t last = 0, idx_size = 0;
  uint64_t dict_total = 0;  // 0 = empty dictionary
  uint64_t dict_base = 0, stats_base = 0;
};

// reads `len` bytes at block offset `off` into dst (host), from host or device memory
int fetch(Ctx* ctx, const uint8_t* blk, bool on_device, uint64_t avail, uint64_t off, void* dst, size_t len) {
  if (off + len > avail) {
    ctx->err = "decode: block runs past the end of the data";
    return ZDWB_ERR_TRUNCATED;
  }
  if (!on_device) {
    memcpy(dst, blk + off, len);
    return ZDWB_OK;
  }
  void* bounce = stage_take(ctx, len);
  if (!bounce) {
    ctx->err = "decode: pinned staging allocation failed";
    return ZDWB_ERR_OOM;
  }
  ZDWB_CUDA_TRY(ctx, cudaMemcpyAsync(bounce, blk + off, len, cudaMemcpyDeviceToHost, ctx->stream));
  ZDWB_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  memcpy(dst, bounce, len);
  return ZDWB_OK;
}

void append_default(std::string& blob, uint8_t type) {  // outputDefault, UnconvertFromZDW.cpp:1224-1266
  if (is_int_type(type)) blob += "0";
  else if (type == ZDWB_DECIMAL) blob += "0.000000000000";
}

// A few bytes from the device to pinned host memory WITHOUT the copy engine: a kernel stores them through the host
// pointer (pinned memory is mapped into the device's address space).  A small cudaMemcpyAsync would queue behind the
// half-gigabyte device->host copy of another context's rows on the same engine - with three contexts taking turns on
// the link every read-back of block k + 1 waited for the rows of block k (end-to-end decode 49 instead of 56 GB/s).
__global__ void k_readback(const uint8_t* __restrict__ src, uint8_t* __restrict__ host_dst, uint32_t n) {
  for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) host_dst[i] = src[i];
}
// (a copy rather than a step of the codec: not counted in Ctx::launches, which stays comparable with earlier runs)
inline cudaError_t readback_small(Ctx* ctx, void* pinned_dst, const void* dev_src, uint32_t n) {
  k_readback<<<1, 128, 0, ctx->stream>>>(static_cast<const uint8_t*>(dev_src), static_cast<uint8_t*>(pinned_dst), n);
  return cudaGetLastError();
}

template <typename T>
int upload(Ctx* ctx, DevBuf& d, const std::vector<T>& v) {
  ZDWB_TRY(d.alloc(ctx, v.size() * sizeof(T) + 16));
  if (!v.empty()) {
    const size_t n = v.size() * sizeof(T);
    void* pinned = stage_take(ctx, n);
    if (!pinned) {
      ctx->err = "decode: pinned staging allocation failed";
      return ZDWB_ERR_OOM;
    }
    memcpy(pinned, v.data(), n);
    ZDWB_CUDA_TRY(ctx, cudaMemcpyAsync(d.p, pinned, n, cudaMemcpyHostToDevice, ctx->stream));
  }
  return ZDWB_OK;
}

// f(std::integral_constant<int, G>) for the lanes per row G = 8, 16 or 32 (anything else: 32), which the row kernels take
// as a template argument
template <class F>
int with_lanes(uint32_t lanes, F f) {
  if (lanes == 8) return f(std::integral_constant<int, 8>());
  if (lanes == 16) return f(std::integral_constant<int, 16>());
  return f(std::integral_constant<int, 32>());
}

// ---------------------------------------------------------------------------------------------
// front end of both decoders (zdwb_decode_block, zdwb_decode_columns): the block header and the used-column tables
// (dec_read_header), the block on the device with the tables and the dictionary's NUL map (dec_upload), the offset of
// every row (dec_find_rows)
// ---------------------------------------------------------------------------------------------
struct DecFront {
  HostBlockHeader H;
  std::vector<uint32_t> used_cols;          // file column of every used column
  std::vector<uint8_t> usz, utype;          // [U]
  std::vector<unsigned long long> ubase;    // [U]
  uint32_t U = 0, F = 0, W = 0, M = 0;
  uint64_t rows_base = 0;
  const uint8_t* src = nullptr;             // the caller's block
  bool in_dev = false;
  uint64_t avail = 0;
  uint64_t win = 0;                         // row-stream bytes on the device
  // (released in reverse order: the buffers a caller allocates afterwards go first)
  DevBuf blk_dev, d_usz, d_ubase, d_utype, d_planes, d_meta, d_nulmap;
  DecParams P;
  DecMeta* meta = nullptr;
};

int dec_read_header(Ctx* ctx, const zdwb_schema* schema, const void* zdw, size_t avail, bool in_dev, DecFront& D) {
  const uint32_t nc = schema->ncols;
  if (nc == 0 || !schema->types) {
    ctx->err = "decode: schema has no columns";
    return ZDWB_ERR_BAD_ARG;
  }
  for (uint32_t c = 0; c < nc; ++c) {
    if (!is_known_type(schema->types[c])) {
      ctx->err = "decode: unsupported column type id " + std::to_string((int)schema->types[c]) + " (v1-v8 files are out of scope)";
      return ZDWB_ERR_UNSUPPORTED;
    }
  }
  const uint8_t* src = static_cast<const uint8_t*>(zdw);
  D.src = src;
  D.in_dev = in_dev;
  D.avail = avail;

  // ---- block header (readLineLength :782-810, readDictionary :812-846, readColumnFieldStats :966-1000)
  HostBlockHeader& H = D.H;
  uint8_t head[16];
  ZDWB_TRY(fetch(ctx, src, in_dev, avail, 0, head, 10));
  memcpy(&H.nrows, head, 4);
  memcpy(&H.line_len, head + 4, 4);
  H.last = head[8];
  H.idx_size = head[9];
  if (H.idx_size > 4) {
    ctx->err = "decode: dictionary index size > 4";
    return ZDWB_ERR_CORRUPT;
  }
  if (H.idx_size) {
    uint8_t tb[4] = {0, 0, 0, 0};
    ZDWB_TRY(fetch(ctx, src, in_dev, avail, 10, tb, H.idx_size));
    uint32_t v;
    memcpy(&v, tb, 4);
    H.dict_total = v;
    H.dict_base = 10 + H.idx_size;
    H.stats_base = H.dict_base + H.dict_total;
  } else {
    H.dict_total = 0;
    H.dict_base = 10;
    H.stats_base = 10;
  }
  std::vector<uint8_t> csize(nc);
  ZDWB_TRY(fetch(ctx, src, in_dev, avail, H.stats_base, csize.data(), nc));
  std::vector<uint32_t>& used_cols = D.used_cols;
  for (uint32_t c = 0; c < nc; ++c)
    if (csize[c]) used_cols.push_back(c);
  const uint32_t U = (uint32_t)used_cols.size();
  D.ubase.assign(U ? U : 1, 0ull);
  if (U) ZDWB_TRY(fetch(ctx, src, in_dev, avail, H.stats_base + nc, D.ubase.data(), (size_t)U * 8));
  D.rows_base = H.stats_base + nc + 8ull * U;
  D.U = U;
  D.F = (U + 7) / 8;
  D.W = (D.F + 3) / 4;
  D.usz.assign(U ? U : 1, 0);
  D.utype.assign(U ? U : 1, 0);
  D.M = D.F;
  for (uint32_t u = 0; u < U; ++u) {
    D.usz[u] = csize[used_cols[u]];
    if (D.usz[u] > 8) {
      ctx->err = "decode: column size > 8";
      return ZDWB_ERR_CORRUPT;
    }
    D.utype[u] = schema->types[used_cols[u]];
    D.M += D.usz[u];
  }
  return ZDWB_OK;
}

int dec_upload(Ctx* ctx, bool at_end_of_file, DecFront& D) {
  cudaStream_t st = ctx->stream;
  const HostBlockHeader& H = D.H;
  const uint32_t U = D.U, F = D.F, W = D.W, M = D.M, nrows = H.nrows;
  const uint64_t rows_base = D.rows_base, avail = D.avail;
  const bool in_dev = D.in_dev;
  const uint8_t* src = D.src;

  // zero-byte rows at the very end of the file are never read by the reference (input->eof(), :1577)
  if (U == 0 && nrows > 0 && at_end_of_file && rows_base >= avail) {
    ctx->err = "Rows unpacked (0) does not match expected (" + std::to_string(nrows) + ")";
    return ZDWB_ERR_ROW_COUNT;
  }

  // ---- residency: the row stream cannot be longer than nrows * M
  const uint64_t win = std::min<uint64_t>(avail > rows_base ? avail - rows_base : 0, (uint64_t)nrows * M);
  if (win >= 0xfffffff0ull) {
    ctx->err = "decode: a block's row stream must be smaller than 4 GiB";
    return ZDWB_ERR_UNSUPPORTED;
  }
  D.win = win;
  const uint8_t* blk;
  if (in_dev) {
    blk = src;
  } else {
    const uint64_t need = rows_base + win;
    ZDWB_TRY(D.blk_dev.alloc(ctx, need + 64));
    if (need >= ((uint64_t)32 << 20) && is_pageable_host(src)) {  // (see encode_block_impl: pageable memory goes through the pinned ring)
      const uint8_t* from = src;
      ZDWB_TRY(ring_h2d(ctx, D.blk_dev.p, (size_t)need, [from](void* dst, size_t off, size_t k) {
        memcpy(dst, from + off, k);
        return true;
      }));
    } else {
      ZDWB_CUDA_TRY(ctx, cudaMemcpyAsync(D.blk_dev.p, src, need, cudaMemcpyHostToDevice, st));
    }
    blk = D.blk_dev.as<uint8_t>();
  }
  const uint64_t dev_avail = in_dev ? avail : rows_base + win;

  // ---- tables
  std::vector<uint32_t> planes((size_t)4 * (W ? W : 1), 0);
  for (uint32_t u = 0; u < U; ++u) {
    for (uint32_t k = 0; k < 4; ++k)
      if (D.usz[u] & (1u << k)) planes[(size_t)k * W + u / 32] |= 1u << (u % 32);
  }
  ZDWB_TRY(upload(ctx, D.d_usz, D.usz));
  ZDWB_TRY(upload(ctx, D.d_ubase, D.ubase));
  ZDWB_TRY(upload(ctx, D.d_utype, D.utype));
  ZDWB_TRY(upload(ctx, D.d_planes, planes));
  ZDWB_TRY(D.d_meta.alloc(ctx, sizeof(DecMeta)));
  ZDWB_CUDA_TRY(ctx, cudaMemsetAsync(D.d_meta.p, 0, sizeof(DecMeta), st));
  D.meta = D.d_meta.as<DecMeta>();

  DecParams& P = D.P;
  P.blk = blk;
  P.avail = dev_avail;
  P.rows_base = rows_base;
  P.dict_base = H.dict_base;
  P.dict_total = H.dict_total;
  P.nrows = nrows;
  P.U = U;
  P.F = F;
  P.M = M;
  P.W = W;
  P.usz = D.d_usz.as<uint8_t>();
  P.ubase = D.d_ubase.as<unsigned long long>();
  P.utype = D.d_utype.as<uint8_t>();
  P.planes = D.d_planes.as<uint32_t>();
  // NUL bitmap of the dictionary: the length of any entry is then one or two word loads
  {
    const uint64_t nwords = (H.dict_total + 31) / 32 + 1;
    ZDWB_TRY(D.d_nulmap.alloc(ctx, nwords * 4));
    ZDWB_TRY(launch(ctx, "k_dict_nulmap", k_dict_nulmap, (unsigned)((nwords + 255) / 256), 256, 0, blk + H.dict_base, H.dict_total,
                    D.d_nulmap.as<uint32_t>(), nwords));
  }
  P.nulmap = D.d_nulmap.as<uint32_t>();
  return ZDWB_OK;
}

// row_off[r] = offset of row r in the row stream (r <= nrows; nrows > 0), found with GL lanes per tile; *consumed_stream =
// where the rows end.  ZDWB_ERR_ROW_COUNT / ZDWB_ERR_TRUNCATED when the data ends before nrows rows do.
int dec_find_rows(Ctx* ctx, const DecFront& D, uint32_t GL, bool at_end_of_file, DevBuf& row_off, uint64_t* consumed_stream) {
  cudaStream_t st = ctx->stream;
  const DecParams& P = D.P;
  const uint32_t nrows = D.H.nrows, U = D.U, M = D.M, W = D.W;
  const uint64_t win = D.win;
  ZDWB_TRY(row_off.alloc(ctx, ((size_t)nrows + 1) * 4));
  *consumed_stream = 0;
  if (U == 0) {
    ZDWB_CUDA_TRY(ctx, cudaMemsetAsync(row_off.p, 0, ((size_t)nrows + 1) * 4, st));
    return ZDWB_OK;
  }
  ZDWB_CUDA_TRY(ctx, cudaMemsetAsync(row_off.p, 0xff, ((size_t)nrows + 1) * 4, st));
  uint32_t T = (uint32_t)std::max<long long>(256, std::min<long long>(ctx->dec_tile_bytes, 32768));
  T &= ~3u;
  // every row occupies at least F bytes, so tiles beyond nrows*M never matter; +1 tile for the end mark
  const uint32_t ntiles = (uint32_t)(win / T) + 1;
  DevBuf maps0;
  ZDWB_TRY(maps0.alloc(ctx, (size_t)ntiles * M * 8));
  const size_t smem_maps = (size_t)T * 4 + ((T + 4 * W + 8) / 4) * 4 + (size_t)4 * W * 4 + 16;
  if (smem_maps > 200 * 1024) {
    ctx->err = "decode: too many used columns for the row-boundary kernel";
    return ZDWB_ERR_UNSUPPORTED;
  }
  ZDWB_CUDA_TRY(ctx, cudaFuncSetAttribute(k_dec_tile_maps, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  ZDWB_TRY(launch(ctx, "k_dec_tile_maps", k_dec_tile_maps, ntiles, DEC_THREADS, smem_maps, P, win, T, maps0.as<uint64_t>()));
  // up-sweep: compose groups of G maps until one remains
  const uint32_t G = 32;
  std::deque<DevBuf> owned;     // the levels above the tile maps and the entry states (a deque: they stay in place)
  std::vector<DevBuf*> levels;  // levels[0] = tile maps
  std::vector<uint32_t> counts;
  levels.push_back(&maps0);
  counts.push_back(ntiles);
  while (counts.back() > 1) {
    const uint32_t n_in = counts.back();
    const uint32_t n_out = (n_in + G - 1) / G;
    DevBuf& nb = owned.emplace_back();
    ZDWB_TRY(nb.alloc(ctx, (size_t)n_out * M * 8));
    ZDWB_TRY(launch(ctx, "k_dec_compose", k_dec_compose, n_out, DEC_THREADS, 0, levels.back()->as<uint64_t>(), n_in, M, G,
                    nb.as<uint64_t>()));
    levels.push_back(&nb);
    counts.push_back(n_out);
  }
  // down-sweep: entry state of every node, from the single root (rows = 0, offset = 0) to the tiles
  DevBuf* ent_parent = &owned.emplace_back();
  ZDWB_TRY(ent_parent->alloc(ctx, 8));
  ZDWB_CUDA_TRY(ctx, cudaMemsetAsync(ent_parent->p, 0, 8, st));
  for (int lv = (int)levels.size() - 2; lv >= 0; --lv) {
    const uint32_t n_in = counts[lv], n_parent = counts[lv + 1];
    DevBuf& ec = owned.emplace_back();
    ZDWB_TRY(ec.alloc(ctx, (size_t)n_in * 8));
    ZDWB_TRY(launch(ctx, "k_dec_descend", k_dec_descend, (n_parent + 127) / 128, 128, 0, levels[lv]->as<uint64_t>(), n_in, M, G,
                    ent_parent->as<uint64_t>(), n_parent, ec.as<uint64_t>()));
    ent_parent = &ec;
  }
  // with a single tile the root entry is the tile entry
  const uint32_t per_cta = DEC_WARPS * (32 / GL);
  const unsigned grid = (ntiles + per_cta - 1) / per_cta;
  ZDWB_TRY(with_lanes(GL, [&](auto g) {
    return launch(ctx, "k_dec_row_starts", k_dec_row_starts<decltype(g)::value>, grid, DEC_THREADS, 0, P, T, ntiles,
                  ent_parent->as<uint64_t>(), row_off.as<uint32_t>());
  }));
  ZDWB_CUDA_TRY(ctx, readback_small(ctx, ctx->meta_host, row_off.as<uint32_t>() + nrows, 4));
  ZDWB_CUDA_TRY(ctx, cudaStreamSynchronize(st));
  const uint32_t h_end = *static_cast<uint32_t*>(ctx->meta_host);
  if (h_end == 0xffffffffu || (uint64_t)h_end > win) {
    // the data ends before `nrows` rows do
    ctx->err = "decode: block truncated (fewer rows than the header promises)";
    return at_end_of_file ? ZDWB_ERR_ROW_COUNT : ZDWB_ERR_TRUNCATED;
  }
  *consumed_stream = h_end;
  return ZDWB_OK;
}

}  // namespace

int decode_block_impl(Ctx* ctx, const zdwb_schema* schema, const void* zdw, size_t avail, const zdwb_decode_opts* opts,
                      zdwb_rows_out* out) {
  memset(out, 0, sizeof(*out));
  ZDWB_TRY(call_begin(ctx));
  cudaStream_t st = ctx->stream;
  DecFront D;
  ZDWB_TRY(dec_read_header(ctx, schema, zdw, avail, opts->input_on_device != 0, D));
  const uint32_t nc = schema->ncols;
  const HostBlockHeader& H = D.H;
  const std::vector<uint32_t>& used_cols = D.used_cols;
  const uint32_t U = D.U, F = D.F;
  out->nrows = H.nrows;
  out->line_length = H.line_len;
  out->is_last = H.last;
  out->dict_bytes = H.dict_total;
  out->ncols_used = U;
  const uint32_t nrows = H.nrows;
  ZDWB_TRY(dec_upload(ctx, opts->at_end_of_file != 0, D));
  const DecParams& P = D.P;
  DecMeta* meta = D.meta;

  // ---- output plan: static segments and dynamic items in output order
  const uint8_t sep = opts->separator;
  const uint8_t term = sep == '\t' ? (uint8_t)'\n' : (uint8_t)0;
  std::vector<int32_t> used_idx(nc, -1);
  for (uint32_t u = 0; u < U; ++u) used_idx[used_cols[u]] = (int32_t)u;
  std::vector<int32_t> pos_src;  // output position -> file column, -1 = blank
  if (opts->out_col) {
    pos_src.assign(opts->n_out, -1);
    for (uint32_t c = 0; c < nc; ++c) {
      const int32_t k = opts->out_col[c];
      if (k < 0) continue;
      if ((uint32_t)k >= opts->n_out) {
        ctx->err = "decode: out_col position out of range";
        return ZDWB_ERR_BAD_ARG;
      }
      pos_src[k] = (int32_t)c;
    }
  } else {
    pos_src.resize(nc);
    for (uint32_t c = 0; c < nc; ++c) pos_src[c] = (int32_t)c;
  }
  std::string blob;
  std::vector<uint32_t> item_u, item_pos, seg_of;  // seg_of[k] = static segment of template byte k
  {
    uint32_t seg = 0;
    for (size_t k = 0; k < pos_src.size(); ++k) {
      if (k) {
        blob.push_back((char)sep);
        seg_of.push_back(seg);
      }
      const int32_t c = pos_src[k];
      if (c < 0) {
        if (opts->out_col && opts->rownum_pos >= 0 && (size_t)opts->rownum_pos == k) {
          item_u.push_back(ITEM_ROWNUM);
          item_pos.push_back((uint32_t)blob.size());
          ++seg;
        } else {
          for (uint32_t f = 0; f < opts->n_fills; ++f) {
            if (opts->fills[f].pos == k && opts->fills[f].len) {
              blob.append(opts->fills[f].text, opts->fills[f].len);
              seg_of.resize(blob.size(), seg);
            }
          }
        }
        continue;
      }
      if (used_idx[c] < 0) {
        append_default(blob, schema->types[c]);
        seg_of.resize(blob.size(), seg);
      } else {
        item_u.push_back((uint32_t)used_idx[c]);
        item_pos.push_back((uint32_t)blob.size());
        ++seg;
      }
    }
    blob.push_back((char)term);
    seg_of.push_back(seg);
  }
  const uint32_t NI = (uint32_t)item_u.size();
  // lanes per row in the row-walking kernels: a whole warp, or 8 / 16 lanes when the schema is narrow enough for every
  // per-row step (flag bytes, output items) to fit one round of that many lanes - a warp then walks 4 / 2 rows at once
  const uint32_t GL = (ctx->dec_group_lanes == 8 || ctx->dec_group_lanes == 16 || ctx->dec_group_lanes == 32)
                          ? (uint32_t)ctx->dec_group_lanes
                          : (NI <= 8 && F <= 8) ? 8u : (NI <= 16 && F <= 16) ? 16u : 32u;
  const uint32_t static_total = (uint32_t)blob.size();
  std::vector<uint4> sgrp;
  for (uint32_t k = 0; k < static_total;) {
    uint32_t n = 1;
    while (n < 4 && k + n < static_total && seg_of[k + n] == seg_of[k]) ++n;
    uint32_t bytes = 0;
    for (uint32_t b2 = 0; b2 < n; ++b2) bytes |= (uint32_t)(uint8_t)blob[k + b2] << (8 * b2);
    sgrp.push_back(make_uint4(bytes, seg_of[k], k, n));
    k += n;
  }
  if (NI >= (1u << 24)) {
    ctx->err = "decode: too many output columns";
    return ZDWB_ERR_UNSUPPORTED;
  }
  DevBuf d_item_u, d_item_pos, d_sgrp;
  ZDWB_TRY(upload(ctx, d_item_u, item_u));
  ZDWB_TRY(upload(ctx, d_item_pos, item_pos));
  ZDWB_TRY(upload(ctx, d_sgrp, sgrp));
  FmtTables FT;
  FT.n_items = NI;
  FT.item_u = d_item_u.as<uint32_t>();
  FT.item_pos = d_item_pos.as<uint32_t>();
  FT.sgrp = d_sgrp.as<uint4>();
  FT.n_groups = (uint32_t)sgrp.size();
  FT.static_total = static_total;
  FT.first_row = opts->first_row_number;
  FT.rownum_item = ITEM_ROWNUM;
  std::vector<int32_t> u_item(U ? U : 1, -1);  // used column -> item (-1: the column is not output)
  for (uint32_t i = 0; i < NI; ++i) {
    if (item_u[i] == ITEM_ROWNUM) FT.rownum_item = i;
    else u_item[item_u[i]] = (int32_t)i;
  }
  DevBuf d_u_item;
  ZDWB_TRY(upload(ctx, d_u_item, u_item));

  if (nrows == 0) {
    out->consumed = D.rows_base;
    return ZDWB_OK;
  }

  // ---- row starts
  DevBuf row_off;
  uint64_t consumed_stream = 0;
  ZDWB_TRY(dec_find_rows(ctx, D, GL, opts->at_end_of_file != 0, row_off, &consumed_stream));
  out->consumed = D.rows_base + consumed_stream;
  if (opts->skim_only) return ZDWB_OK;  // the caller only wanted to know where the next block starts

  // ---- strips: one warp walks RS consecutive rows (k_dec_rows); about four waves of warps over the GPU
  if (U >= (1u << 24) || NI >= (1u << 24)) {
    ctx->err = "decode: more than 2^24 used columns";
    return ZDWB_ERR_UNSUPPORTED;
  }
  // about 48 strips per SM (two waves of the 24 resident warps), rounded down to a power of two: measured on C4,
  // 16- and 32-row strips run 7-25 % faster than 18, 24 or 40 (profiles/README.md)
  // lanes per strip in the row kernels: a whole warp, or 8 / 16 lanes when the schema is narrow enough for every
  // per-row step (flag bytes, output items) to fit one round of that many lanes
  const uint32_t G = GL;
  const uint32_t GPW = 32 / G;
  // ---- the delta writer takes wide schemas whose output order follows the file order (so that the changed items of a
  // row come out of the flag walk in output order) and no running row number
  bool use_delta = ctx->dec_delta != 0 && GL == 32 && FT.rownum_item == ITEM_ROWNUM && NI > 0 && NI < 32768 && U < 65536;
  {
    int32_t last_item = -1;
    for (uint32_t u = 0; u < U && use_delta; ++u) {
      if (u_item[u] < 0) continue;
      if (u_item[u] <= last_item) use_delta = false;
      last_item = u_item[u];
    }
  }
  uint32_t R = 8;
  // (the delta writer starts every strip with a row assembled in full: it likes strips twice as long - measured on C4:
  // 0.79 ms with 16 rows, 0.74 with 32, 1.27 with 64)
  while (R < 64 && (uint64_t)R * 2 <= nrows / ((uint64_t)ctx->sm_count * (use_delta ? 24 : 48) * GPW)) R *= 2;
  // (a block of a few thousand rows: shorter strips until there are some sixteen warps per SM - measured on the
  // 3768-row C3 golden: 0.79 ms with 8-row strips, 0.68 with 4, 0.64 with 2)
  while (R > 2 && nrows / R < (uint64_t)ctx->sm_count * 16 * GPW) R /= 2;
  if (ctx->dec_strip_rows > 0) R = (uint32_t)ctx->dec_strip_rows;
  const uint32_t nstrips = (nrows + R - 1) / R;

  DevBuf cin, d_counts;
  ZDWB_TRY(cin.alloc(ctx, (size_t)nstrips * std::max(U, 1u) * 8));
  if (opts->want_flag_counts && U) {
    ZDWB_TRY(d_counts.alloc(ctx, (size_t)U * 8));
    ZDWB_CUDA_TRY(ctx, cudaMemsetAsync(d_counts.p, 0, (size_t)U * 8, st));
  }
  if (U == 0 && opts->validate_only) return ZDWB_OK;
  if (U) {
    DevBuf sval, shas;
    ZDWB_TRY(sval.alloc(ctx, (size_t)nstrips * U * 8));
    ZDWB_TRY(shas.alloc(ctx, (size_t)nstrips * U));
    const size_t smem_sum = (size_t)U * 4 + 16;
    ZDWB_TRY(with_lanes(GL, [&](auto g) -> int {
      auto k = k_dec_strip_summary<decltype(g)::value>;
      ZDWB_CUDA_TRY(ctx, cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      return launch(ctx, "k_dec_strip_summary", k, nstrips, DEC_THREADS, smem_sum, P, row_off.as<uint32_t>(), R, opts->validate_only,
                    d_counts.as<unsigned long long>(), sval.as<unsigned long long>(), shas.as<uint8_t>(), meta);
    }));
    if (opts->validate_only || opts->want_flag_counts) {
      DecMeta* hm0 = static_cast<DecMeta*>(ctx->meta_host);
      ZDWB_CUDA_TRY(ctx, cudaMemcpyAsync(hm0, meta, sizeof(DecMeta), cudaMemcpyDeviceToHost, st));
      if (opts->want_flag_counts) {
        ctx->flag_counts.resize(U);
        ZDWB_CUDA_TRY(ctx, cudaMemcpyAsync(ctx->flag_counts.data(), d_counts.p, (size_t)U * 8, cudaMemcpyDeviceToHost, st));
      }
      ZDWB_CUDA_TRY(ctx, cudaStreamSynchronize(st));
      if (opts->want_flag_counts) out->flag_counts = reinterpret_cast<const uint64_t*>(ctx->flag_counts.data());
      if (opts->validate_only) {
        if (hm0->err) {
          ctx->err = "decode: dictionary offset out of range";
          return ZDWB_ERR_CORRUPT;  // CORRUPTED_DATA_ERROR, UnconvertFromZDW.cpp:1532-1534
        }
        return ZDWB_OK;
      }
    }
    ZDWB_TRY(carry_prefix(ctx, sval.as<unsigned long long>(), shas.as<uint8_t>(), nstrips, U, cin.as<unsigned long long>()));
  }

  // ---- shared-memory layout of a warp in k_dec_rows: lengths-only pass and writing pass
  auto make_layout = [&](bool write, WarpLayout& L) -> bool {
    const size_t NIe = std::max(NI, 1u);
    size_t o = 0;
    L.o_len = (uint32_t)o;    o += NIe * 4;
    o = (o + 7) & ~(size_t)7;
    L.o_val = (uint32_t)o;    if (write) o += NIe * 4;
    o = (o + 15) & ~(size_t)15;
    L.o_textc = (uint32_t)o;  if (write) o += NIe * 16;
    L.o_ioff = (uint32_t)o;   o += ((size_t)NI + 1) * 4;
    L.o_llist = (uint32_t)o;  o += (1 + (size_t)NI) * 4;
    o = (o + 15) & ~(size_t)15;
    if (o > 200 * 1024) return false;
    // L.stride = bytes of one strip group's state; a CTA holds L.warps * GPW of them
    uint32_t warps = 4;
    while (warps > 1 && o * warps * GPW > 200 * 1024) warps >>= 1;
    L.warps = warps;
    L.stride = (uint32_t)o;
    return (size_t)L.stride * warps * GPW <= 200 * 1024;
  };
  WarpLayout L1, L2;
  if (!make_layout(false, L1) || !make_layout(true, L2)) {
    ctx->err = "decode: too many used columns for the row kernels";
    return ZDWB_ERR_UNSUPPORTED;
  }

  // ---- pass A: length of every row, then the row offsets and the exact output size
  ctx->out_dev2 = nullptr;
  {
    DevBuf ro;
    ZDWB_TRY(ro.alloc(ctx, ((size_t)nrows + 1) * 8));
    ctx->out_dev2 = ro.detach();
  }
  unsigned long long* d_row_off = static_cast<unsigned long long*>(ctx->out_dev2);
  DevBuf row_len;
  ZDWB_TRY(row_len.alloc(ctx, (size_t)nrows * 8));
  // k_dec_rows, timed as `name`: lengths only (write = false) or the rows
  auto launch_rows = [&](const char* name, bool write, const WarpLayout& L, unsigned long long* lens, const unsigned long long* offs,
                         uint8_t* dst) -> int {
    const uint32_t per_cta = L.warps * GPW;
    const unsigned grid = (nstrips + per_cta - 1) / per_cta, block = 32 * L.warps;
    const size_t smem = (size_t)L.stride * per_cta;
    return with_lanes(G, [&](auto g) -> int {
      auto k = write ? k_dec_rows<true, decltype(g)::value> : k_dec_rows<false, decltype(g)::value>;
      ZDWB_CUDA_TRY(ctx, cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, 208 * 1024));
      return launch(ctx, name, k, grid, block, smem, P, FT, d_u_item.as<int32_t>(), row_off.as<uint32_t>(), R, L,
                    cin.as<unsigned long long>(), lens, offs, dst, meta);
    });
  };
  ZDWB_TRY(launch_rows("k_dec_row_lens", false, L1, row_len.as<unsigned long long>(), nullptr, nullptr));
  ZDWB_TRY(exclusive_scan_u64(ctx, reinterpret_cast<const uint64_t*>(row_len.p), reinterpret_cast<uint64_t*>(d_row_off), nrows,
                              reinterpret_cast<uint64_t*>(d_row_off + nrows)));
  DecMeta* hm = static_cast<DecMeta*>(ctx->meta_host);
  ZDWB_CUDA_TRY(ctx, readback_small(ctx, hm, meta, (uint32_t)sizeof(DecMeta)));
  ZDWB_CUDA_TRY(ctx, readback_small(ctx, reinterpret_cast<uint8_t*>(ctx->meta_host) + 1024, d_row_off + nrows, 8));
  ZDWB_CUDA_TRY(ctx, cudaStreamSynchronize(st));
  if (hm->err) {
    ctx->err = "decode: dictionary offset out of range";
    return ZDWB_ERR_CORRUPT;  // CORRUPTED_DATA_ERROR, UnconvertFromZDW.cpp:1364-1365
  }
  memcpy(&hm->out_bytes, reinterpret_cast<uint8_t*>(ctx->meta_host) + 1024, 8);
  ctx->last_out_per_row = hm->out_bytes / nrows;

  // ---- pass B: the rows
  ctx->out_dev = nullptr;
  {
    // (64 bytes in front: the delta writer's merged chunks may read up to 15 bytes in front of the first row)
    DevBuf ob;
    ZDWB_TRY(ob.alloc(ctx, hm->out_bytes + 192));
    ctx->out_dev = static_cast<uint8_t*>(ob.detach()) + 64;
  }
  if (use_delta) {
    // per-warp state of the delta writer: column values, lengths, their prefix, the lists of a row's changed items
    DeltaLayout DL;
    size_t o = 0;
    DL.o_val = (uint32_t)o;    o += (size_t)NI * 8;
    DL.o_len = (uint32_t)o;    o += (size_t)NI * 4;
    DL.o_ioff = (uint32_t)o;   o += ((size_t)NI + 1) * 4;
    DL.o_lcs = (uint32_t)o;    o += (size_t)DLC * 4;
    DL.o_lce = (uint32_t)o;    o += (size_t)DLC * 4;
    DL.o_lpe = (uint32_t)o;    o += (size_t)DLC * 4;
    DL.o_lvoff = (uint32_t)o;  o += (size_t)DLC * 4;
    DL.o_litem = (uint32_t)o;  o += (size_t)DLC * 2;
    DL.o_lu = (uint32_t)o;     o += (size_t)DLC * 2;
    DL.o_slow = (uint32_t)o;   o += std::max<size_t>(2 * DLC + 4, NI) * 2;
    o = (o + 15) & ~(size_t)15;
    uint32_t warps = 4;
    while (warps > 1 && o * warps > 200 * 1024) warps >>= 1;
    if (o * warps > 200 * 1024) {
      use_delta = false;
    } else {
      DL.stride = (uint32_t)o;
      DL.warps = warps;
      std::vector<uint8_t> outmask((size_t)F + 4, 0);
      for (uint32_t u = 0; u < U; ++u)
        if (u_item[u] >= 0) outmask[u >> 3] |= (uint8_t)(1u << (u & 7u));
      DevBuf d_outmask;
      ZDWB_TRY(upload(ctx, d_outmask, outmask));
      ZDWB_CUDA_TRY(ctx, cudaFuncSetAttribute(k_dec_write_delta, cudaFuncAttributeMaxDynamicSharedMemorySize, 208 * 1024));
      const unsigned grid = (nstrips + warps - 1) / warps;
      ZDWB_TRY(launch(ctx, "k_dec_write_delta", k_dec_write_delta, grid, 32 * warps, (size_t)DL.stride * warps, P, FT,
                      d_u_item.as<int32_t>(), d_outmask.as<uint8_t>(), row_off.as<uint32_t>(), R, DL, cin.as<unsigned long long>(),
                      d_row_off, static_cast<uint8_t*>(ctx->out_dev), meta));
    }
  }
  if (!use_delta) ZDWB_TRY(launch_rows("k_dec_write_rows", true, L2, nullptr, d_row_off, static_cast<uint8_t*>(ctx->out_dev)));
  const uint64_t out_len = hm->out_bytes;
  out->len = out_len;
  if (opts->output_on_device) {
    ZDWB_CUDA_TRY(ctx, cudaStreamSynchronize(st));
    out->tsv = static_cast<const uint8_t*>(ctx->out_dev);
    out->row_off = opts->want_row_offsets ? static_cast<const uint64_t*>(ctx->out_dev2) : nullptr;
    return ZDWB_OK;
  }
  // Pinning memory costs about as much as copying into it a few times over: worth it when more blocks follow and re-use
  // the buffer, not for a context whose first block is also the file's last - that one result goes to plain memory.
  // (measured: 0.45 s per GiB pinned, serialised with every other context's driver calls, against ~0.1 s per GiB for a
  // copy into pageable memory - so the first results of a context go to plain memory as well)
  const bool one_off = (ctx->decode_calls == 0 && H.last) || ctx->decode_calls < 3;
  ++ctx->decode_calls;
  if (ctx->out_host_cap < out_len || (!ctx->out_host_pinned && !one_off)) {
    out_host_release(ctx);
    if (one_off) {
      ctx->out_host = malloc(out_len + out_len / 8 + 64);
      if (!ctx->out_host) {
        ctx->err = "decode: host allocation failed";
        return ZDWB_ERR_OOM;
      }
      ctx->out_host_pinned = false;
      ctx->out_host_cap = out_len + out_len / 8;
    } else {
      const size_t cap = std::max<size_t>(out_len + out_len / 4, 1 << 20);  // headroom: blocks of a file vary a little
      ZDWB_CUDA_TRY(ctx, cudaHostAlloc(&ctx->out_host, cap, cudaHostAllocDefault));
      ctx->out_host_pinned = true;
      ctx->out_host_cap = cap;
    }
  }
  if (!ctx->out_host_pinned && out_len >= ((size_t)32 << 20)) {
    // a plain host buffer: through the pinned ring, chunk by chunk (the driver's own staging is several times slower)
    uint8_t* dst = static_cast<uint8_t*>(ctx->out_host);
    ZDWB_TRY(ring_d2h(ctx, ctx->out_dev, out_len, [dst](const uint8_t* src, size_t off, size_t k) {
      memcpy(dst + off, src, k);
      return true;
    }));
  } else if (ctx->copy_gate && out_len >= COPY_GATE_MIN) {
    ZDWB_CUDA_TRY(ctx, cudaStreamSynchronize(st));  // the rows are written: now wait for the link, not with it
    std::lock_guard<std::mutex> turn(copy_gate(ctx->device, 1));
    ZDWB_CUDA_TRY(ctx, cudaMemcpyAsync(ctx->out_host, ctx->out_dev, out_len, cudaMemcpyDeviceToHost, st));
    ZDWB_CUDA_TRY(ctx, cudaStreamSynchronize(st));
  } else {
    ZDWB_CUDA_TRY(ctx, cudaMemcpyAsync(ctx->out_host, ctx->out_dev, out_len, cudaMemcpyDeviceToHost, st));
  }
  if (opts->want_row_offsets) {
    const size_t rb = ((size_t)nrows + 1) * 8;
    if (ctx->out_host2_cap < rb) {
      if (ctx->out_host2) cudaFreeHost(ctx->out_host2);
      ctx->out_host2 = nullptr;
      ctx->out_host2_cap = 0;
      ZDWB_CUDA_TRY(ctx, cudaHostAlloc(&ctx->out_host2, std::max<size_t>(rb + rb / 4, 1 << 16), cudaHostAllocDefault));
      ctx->out_host2_cap = std::max<size_t>(rb + rb / 4, 1 << 16);
    }
    ZDWB_CUDA_TRY(ctx, cudaMemcpyAsync(ctx->out_host2, ctx->out_dev2, rb, cudaMemcpyDeviceToHost, st));
    out->row_off = static_cast<const uint64_t*>(ctx->out_host2);
  }
  ZDWB_CUDA_TRY(ctx, cudaStreamSynchronize(st));
  out->tsv = static_cast<const uint8_t*>(ctx->out_host);
  return ZDWB_OK;
}


int decode_columns_impl(Ctx* ctx, const zdwb_schema* schema, const void* zdw, size_t avail, const zdwb_columns_opts* opts,
                        zdwb_columns_out* out) {
  memset(out, 0, sizeof(*out));
  ZDWB_TRY(call_begin(ctx));
  cudaStream_t st = ctx->stream;
  const uint32_t nc = schema->ncols, K = opts->n_cols;
  if (K == 0 || !opts->cols) {
    ctx->err = "decode_columns: empty column list";
    return ZDWB_ERR_BAD_ARG;
  }
  {
    std::vector<uint8_t> seen(nc, 0);
    for (uint32_t k = 0; k < K; ++k) {
      const uint32_t c = opts->cols[k];
      if (c >= nc) {
        ctx->err = "decode_columns: column index " + std::to_string(c) + " out of range (the schema has " + std::to_string(nc) + ")";
        return ZDWB_ERR_BAD_ARG;
      }
      if (seen[c]) {
        ctx->err = "decode_columns: column " + std::to_string(c) + " listed twice";
        return ZDWB_ERR_BAD_ARG;
      }
      seen[c] = 1;
    }
  }
  DecFront D;
  ZDWB_TRY(dec_read_header(ctx, schema, zdw, avail, opts->input_on_device != 0, D));
  const HostBlockHeader& H = D.H;
  const uint32_t U = D.U, F = D.F, nrows = H.nrows;
  out->nrows = nrows;
  out->line_length = H.line_len;
  out->is_last = H.last;
  out->dict_bytes = H.dict_total;
  out->ncols_used = U;
  ZDWB_TRY(dec_upload(ctx, opts->at_end_of_file != 0, D));
  const DecParams& P = D.P;

  // ---- the selected used columns in ascending order (sel_u) with their output rows (sel_k); unused ones are filled
  std::vector<int32_t> used_idx(nc, -1);
  for (uint32_t u = 0; u < U; ++u) used_idx[D.used_cols[u]] = (int32_t)u;
  std::vector<std::pair<uint32_t, uint32_t>> sel;
  bool want_dict = false;
  for (uint32_t k = 0; k < K; ++k) {
    const uint32_t c = opts->cols[k];
    if (is_text_like(schema->types[c])) want_dict = true;
    if (used_idx[c] >= 0) sel.emplace_back((uint32_t)used_idx[c], k);
  }
  std::sort(sel.begin(), sel.end());
  std::vector<uint32_t> sel_u(sel.size()), sel_k(sel.size());
  for (size_t j = 0; j < sel.size(); ++j) {
    sel_u[j] = sel[j].first;
    sel_k[j] = sel[j].second;
  }

  // ---- outputs: the values, and with a text-like column the dictionary and where its entries start
  unsigned long long* values;
  {
    DevBuf vb;
    ZDWB_TRY(vb.alloc(ctx, (size_t)K * nrows * 8 + 16));
    values = static_cast<unsigned long long*>(vb.detach());
  }
  const uint64_t nwords = (H.dict_total + 31) / 32 + 1;  // words of the NUL map
  DevBuf dict_prefix;
  uint32_t* h_entries = reinterpret_cast<uint32_t*>(static_cast<uint8_t*>(ctx->meta_host) + 2048);
  if (want_dict) {
    DevBuf db;
    ZDWB_TRY(db.alloc(ctx, H.dict_total + 16));
    if (H.dict_total) ZDWB_CUDA_TRY(ctx, cudaMemcpyAsync(db.p, P.blk + H.dict_base, H.dict_total, cudaMemcpyDeviceToDevice, st));
    out->dict = static_cast<const uint8_t*>(db.detach());
    DevBuf d_total;
    ZDWB_TRY(d_total.alloc(ctx, 4));
    ZDWB_TRY(dict_prefix.alloc(ctx, nwords * 4));
    ZDWB_TRY(launch(ctx, "k_dict_counts", k_dict_counts, (unsigned)((nwords + 255) / 256), 256, 0, P.nulmap, H.dict_total,
                    dict_prefix.as<uint32_t>(), nwords));
    ZDWB_TRY(exclusive_scan_u32(ctx, dict_prefix.as<uint32_t>(), dict_prefix.as<uint32_t>(), nwords, d_total.as<uint32_t>()));
    ZDWB_CUDA_TRY(ctx, cudaMemcpyAsync(h_entries, d_total.p, 4, cudaMemcpyDeviceToHost, st));
  }

  // ---- row starts: lanes per row by the width of the flag bytes, as in zdwb_decode_block
  const uint32_t GL = (ctx->dec_group_lanes == 8 || ctx->dec_group_lanes == 16 || ctx->dec_group_lanes == 32)
                          ? (uint32_t)ctx->dec_group_lanes
                          : F <= 8 ? 8u : F <= 16 ? 16u : 32u;
  DevBuf row_off;
  uint64_t consumed_stream = 0;
  if (nrows) ZDWB_TRY(dec_find_rows(ctx, D, GL, opts->at_end_of_file != 0, row_off, &consumed_stream));
  out->consumed = D.rows_base + consumed_stream;

  if (want_dict) {
    ZDWB_CUDA_TRY(ctx, cudaStreamSynchronize(st));  // (the number of entries)
    const uint64_t n = *h_entries;
    DevBuf eb;
    ZDWB_TRY(eb.alloc(ctx, (n + 1) * 8));
    ZDWB_TRY(launch(ctx, "k_dict_entries", k_dict_entries, (unsigned)((nwords + 255) / 256), 256, 0, P.nulmap, H.dict_total,
                    dict_prefix.as<uint32_t>(), nwords, eb.as<unsigned long long>()));
    out->entry_off = static_cast<const uint64_t*>(eb.detach());
    out->dict_entries = n;
  }
  if (nrows) {
    // a column the block does not use holds its type's default in every row
    for (uint32_t k = 0; k < K; ++k) {
      const uint32_t c = opts->cols[k];
      if (used_idx[c] < 0)
        ZDWB_CUDA_TRY(ctx, cudaMemsetAsync(values + (size_t)k * nrows, is_text_like(schema->types[c]) ? 0xff : 0, (size_t)nrows * 8, st));
    }
  }
  if (nrows && !sel.empty()) {
    // ---- strips of 32 rows: the value every used column holds where a strip begins, then one warp per strip
    const uint32_t R = 32, nstrips = (nrows + R - 1) / R;
    DevBuf cin, sval, shas, d_sel_u, d_sel_k;
    ZDWB_TRY(cin.alloc(ctx, (size_t)nstrips * U * 8));
    ZDWB_TRY(sval.alloc(ctx, (size_t)nstrips * U * 8));
    ZDWB_TRY(shas.alloc(ctx, (size_t)nstrips * U));
    const size_t smem_sum = (size_t)U * 4 + 16;
    ZDWB_TRY(with_lanes(GL, [&](auto g) -> int {
      auto k = k_dec_strip_summary<decltype(g)::value>;
      ZDWB_CUDA_TRY(ctx, cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      return launch(ctx, "k_dec_strip_summary", k, nstrips, DEC_THREADS, smem_sum, P, row_off.as<uint32_t>(), R, 0,
                    (unsigned long long*)nullptr, sval.as<unsigned long long>(), shas.as<uint8_t>(), D.meta);
    }));
    ZDWB_TRY(carry_prefix(ctx, sval.as<unsigned long long>(), shas.as<uint8_t>(), nstrips, U, cin.as<unsigned long long>()));
    ZDWB_TRY(upload(ctx, d_sel_u, sel_u));
    ZDWB_TRY(upload(ctx, d_sel_k, sel_k));
    ZDWB_TRY(launch(ctx, "k_dec_columns", k_dec_columns, (nstrips + DEC_WARPS - 1) / DEC_WARPS, DEC_THREADS, 0, P,
                    row_off.as<uint32_t>(), cin.as<unsigned long long>(), d_sel_u.as<uint32_t>(), d_sel_k.as<uint32_t>(),
                    (uint32_t)sel.size(), dict_prefix.as<uint32_t>(), values, D.meta));
  }
  DecMeta* hm = static_cast<DecMeta*>(ctx->meta_host);
  ZDWB_CUDA_TRY(ctx, cudaMemcpyAsync(hm, D.meta, sizeof(DecMeta), cudaMemcpyDeviceToHost, st));
  ZDWB_CUDA_TRY(ctx, cudaStreamSynchronize(st));
  if (hm->err) {
    ctx->err = "decode_columns: a text value's dictionary offset is not the start of an entry";
    return ZDWB_ERR_CORRUPT;
  }
  out->values = reinterpret_cast<const int64_t*>(values);
  return ZDWB_OK;
}

}  // namespace zdwb
