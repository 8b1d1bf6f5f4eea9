// encode.cu -- TSV -> one ZDW block, entirely on the GPU.
//
// Kernel sequence for a block (reference functions replaced are cited per kernel):
//   k_tile_count, k_tile_scan     GetNextRow + get_next_column as a byte-tile census: row terminators, field separators,
//                                 non-empty fields per 16 KiB tile and their prefix over the buffer
//                                 (getnextrow.cpp:26-84, ConvertToZDW.cpp:1048-1067)
//   k_find_cut                    block cut after max_rows rows (explicit block policy)
//   k_pass1                       parseInput (ConvertToZDW.cpp:329-414) + Dictionary::insert (dictionary.cpp:31-51):
//                                 one warp per tile, no CTA barrier; the non-empty fields of a 512-byte step go to a
//                                 warp-private queue (slot = ordinal) and are worked off 32 at a time: numbers and CHAR
//                                 cells at once from registers, texts parked in two side queues by length and inserted
//                                 into the hash set 32 of a kind at a time; a compact RECORD (column, dictionary slot or
//                                 number) per non-empty field is written in row order, so pass 2 never re-reads or
//                                 re-parses the TSV
//   k_ht_compact, sort_strings, k_sorted_lens, k_dict_slots, k_dict_emit
//                                 Dictionary::write              dictionary.cpp:76-111
//   k_col_stats, k_col_info, k_block_header   writeLookupColumnStats         ConvertToZDW.cpp:417-483, :839-842
//   k_pass2, k_gather_tiles       writeBlockRows                 ConvertToZDW.cpp:486-606 + Dictionary::getOffset :53-59
//   k_p2d_rowlen, k_p2d_emit      the same for the row-delta path, from each row's own records
//
// Data layout in HBM: the TSV block is read twice (census, pass 1; the census-free row-delta pass 1 reads it once);
// records are 12 B per NON-EMPTY field (most fields of analytics-shaped data are empty and cost nothing beyond their
// delimiter byte); the string hash set keeps (start, len) of the first occurrence inside the TSV - strings are never
// copied until the dictionary is emitted.
#include <algorithm>
#include <vector>

#include "common.cuh"

namespace zdwb {

namespace {

constexpr int ENC_THREADS = 256;
constexpr int ENC_WARPS = ENC_THREADS / 32;
constexpr uint32_t TILE = 16384;          // bytes per warp tile
constexpr uint32_t STEP = 512;            // bytes per warp step (32 lanes x 16 B)
constexpr uint32_t HT_MAX_PROBE = 2048;
constexpr uint32_t SHORT_MAX = 16;        // texts up to this length are hashed / compared by one lane, straight-line
constexpr uint32_t REC_EMPTY = 0xffffffffu;
// row-delta records: rec_col bit 31 = the value equals the row before's (no repeat flag); columns are < 4096 there
constexpr uint32_t REC_SAME = 1u << 31;

struct EncMeta {
  uint32_t bad_row;        // first row whose field count != schema (0xffffffff = none)
  uint32_t max_line;       // longest logical line incl. '\n' among the block's rows (+ tail rule)
  uint32_t ht_overflow;    // pass 1 gave up: hash table too small
  uint32_t pad1;
  unsigned long long n_unique;
  unsigned long long dict_str_bytes;  // sum(len + 1)
  uint32_t max_str_len;
  uint32_t n_used;
  uint32_t idx_size;
  uint32_t nflag;
  uint32_t max_row_bytes;
  uint32_t pad0;
  uint64_t dict_total;   // Dictionary::getSize()
  uint64_t dict_base;    // offset of the dictionary origin byte inside the block
  uint64_t stats_base;
  uint64_t rows_base;
  unsigned long long rows_bytes;
  uint32_t compact_count;
  uint32_t rec_count;      // delta path: records handed out so far (atomic bump allocator)
  uint32_t rec_overflow;   // ... the record arrays were too small: retry with larger ones
  uint32_t delta_bail;     // ... a row does not fit the warp's lists: the block goes through the general pass 1
  // census totals
  uint32_t tot_rows, tot_tabs, tot_ne, last_break_p1;
  // block cut (max_rows)
  uint32_t cut_end_p1;     // position + 1 of the terminator of the block's last row
  uint32_t next_start;     // first byte of the row after it
  uint32_t spill_end;      // position + 1 of the delimiter that closes the last spilled column of that row
  uint32_t spill_row_len;  // length of that row incl. its terminator (0 = there is no complete row)
  // census-free row-delta pass 1 (k_pass1d<true>): rows are numbered per tile, k_row_fixup makes the numbers global
  uint32_t slot_overflow;  // a tile owns more rows than it has slots: the block is run again with the census
  uint32_t pad2;
  unsigned long long bad_slot;  // (tile << 32) | row of the tile, of the first malformed row (~0 = none)
};

// per tile: counts, then (after k_tile_scan) exclusive prefixes
struct TileAgg {
  uint32_t rows, tabs, ne;
  uint32_t bound_p1;   // position + 1 of the last boundary (separator, terminator, blank-line newline); 0 = none
  uint32_t break_p1;   // position + 1 of the last row break (terminator or blank-line newline); 0 = none
  uint32_t rs_p1;      // position + 1 of the last row START (first byte of a non-blank line); 0 = none.  Only the
                       // row census of the delta path (k_row_census) fills it in
};

// ---------------------------------------------------------------------------------------------
// byte classification, one warp step = 512 bytes.
//
// Rules restated from the reference (SURVEY Appendix B-2, B-3):
//  * '\n' ends a logical row iff it is preceded by an EVEN number of consecutive backslashes
//    (GetNextRow, getnextrow.cpp:44-53,72-77);
//  * '\t' separates fields iff it is preceded by an EVEN number of consecutive backslashes
//    (get_next_column, ConvertToZDW.cpp:1048-1067); a maximal-run count reproduces the reference's bounded backward
//    scans because a delimiter byte itself is never a backslash;
//  * an unescaped newline directly after another unescaped newline (or at offset 0) is a blank physical line and
//    ends no row (getnextrow.cpp:39-43).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ bool odd_backslashes_before(const uint8_t* __restrict__ buf, int64_t p) {
  uint32_t c = 0;
  int64_t q = p - 1;
  while (q >= 0 && __ldg(buf + q) == (uint8_t)'\\') {
    ++c;
    --q;
  }
  return (c & 1u) != 0;
}
__device__ __forceinline__ bool is_unescaped_newline(const uint8_t* __restrict__ buf, int64_t p) {
  return __ldg(buf + p) == (uint8_t)'\n' && !odd_backslashes_before(buf, p);
}

struct WarpCarry {
  uint32_t bs;      // the byte in front of the step is a backslash
  uint32_t nl;      // ... is an unescaped newline (or the step starts at offset 0)
  int64_t pb;       // position of the last boundary in front of the step (-1 = buffer start)
  int64_t prb;      // position of the last row break in front of the step (-1 = buffer start)
  uint32_t rows, tabs, ne;  // running counts in front of the step
};

struct LaneStep {
  uint32_t tab, term, skip;  // 16-bit masks for the lane's 16 bytes
  uint32_t ne;               // delimiters that close a non-empty field
  int64_t p0;                // position of the lane's first byte (may be negative / beyond n: masks are then empty)
  int64_t pb, prb;           // last boundary / row break in front of the lane's chunk
  uint32_t rows, tabs, nes;  // counts in front of the lane's chunk
};

__device__ __forceinline__ void carry_init(const uint8_t* __restrict__ buf, int64_t p, const TileAgg& pre, WarpCarry& c) {
  c.bs = (p > 0 && __ldg(buf + p - 1) == (uint8_t)'\\') ? 1u : 0u;
  c.nl = p <= 0 ? 1u : (is_unescaped_newline(buf, p - 1) ? 1u : 0u);
  c.pb = (int64_t)pre.bound_p1 - 1;
  c.prb = (int64_t)pre.break_p1 - 1;
  c.rows = pre.rows;
  c.tabs = pre.tabs;
  c.ne = pre.ne;
}

// Classifies the 512 bytes at step position s0 (s0 + 16 * lane is 16-byte aligned in memory).  Only positions in
// [0, limit) are reported.  All 32 lanes must call.
__device__ __forceinline__ LaneStep scan_step(const uint8_t* __restrict__ buf, int64_t limit, int64_t s0, WarpCarry& c) {
  const unsigned lane = lane_id();
  LaneStep L;
  L.p0 = s0 + 16 * (int64_t)lane;
  uint32_t tab = 0, nl = 0, bs = 0;
  if (L.p0 < limit && L.p0 + 16 > 0) {
    const uint4 v = ldg_stream_u4(buf + L.p0);
    const int64_t ia = L.p0 < 0 ? -L.p0 : 0;
    const int64_t ib = L.p0 + 16 > limit ? limit - L.p0 : 16;
    const uint32_t in = ((1u << ib) - 1u) & ~((1u << ia) - 1u);
    tab = chunk_mask(v, '\t') & in;
    if (chunk_has(v, '\n')) nl = chunk_mask(v, '\n') & in;
    if (chunk_has(v, '\\')) bs = chunk_mask(v, '\\') & in;
  }
  // escape parity: only delimiters that directly follow a backslash need the (rare) backward walk
  uint32_t prev = __shfl_up_sync(0xffffffffu, bs >> 15, 1);
  if (lane == 0) prev = c.bs;
  uint32_t sus = (tab | nl) & ((bs << 1) | prev);
  while (sus) {
    const int i = __ffs(sus) - 1;
    sus &= sus - 1;
    if (odd_backslashes_before(buf, L.p0 + i)) {
      tab &= ~(1u << i);
      nl &= ~(1u << i);
    }
  }
  // blank lines
  uint32_t prevnl = __shfl_up_sync(0xffffffffu, nl >> 15, 1);
  if (lane == 0) prevnl = c.nl;
  uint32_t after_nl = ((nl << 1) | prevnl) & 0xffffu;
  if (L.p0 <= 0 && L.p0 + 16 > 0) after_nl |= 1u << (-L.p0);  // offset 0 behaves like "just after a newline"
  L.tab = tab;
  L.skip = nl & after_nl;
  L.term = nl & ~L.skip;
  c.bs = __shfl_sync(0xffffffffu, bs >> 15, 31);
  c.nl = __shfl_sync(0xffffffffu, nl >> 15, 31);

  // nearest boundary / row break in front of the lane's chunk: from the closest lower lane that has one
  const uint32_t bound = L.tab | L.term | L.skip, brk = L.term | L.skip;
  const int64_t mylast_b = bound ? L.p0 + (31 - __clz(bound)) : 0;
  const int64_t mylast_r = brk ? L.p0 + (31 - __clz(brk)) : 0;
  const unsigned has_b = __ballot_sync(0xffffffffu, bound != 0u), has_r = __ballot_sync(0xffffffffu, brk != 0u);
  const unsigned lt = lanemask_lt();
  {
    const unsigned below = has_b & lt;
    const int64_t v = __shfl_sync(0xffffffffu, mylast_b, below ? 31 - __clz(below) : 0);
    L.pb = below ? v : c.pb;
    const int64_t top = __shfl_sync(0xffffffffu, mylast_b, has_b ? 31 - __clz(has_b) : 0);
    if (has_b) c.pb = top;
  }
  {
    const unsigned below = has_r & lt;
    const int64_t v = __shfl_sync(0xffffffffu, mylast_r, below ? 31 - __clz(below) : 0);
    L.prb = below ? v : c.prb;
    const int64_t top = __shfl_sync(0xffffffffu, mylast_r, has_r ? 31 - __clz(has_r) : 0);
    if (has_r) c.prb = top;
  }
  // delimiters whose preceding byte is not a boundary close a non-empty field
  const uint32_t delims = L.tab | L.term;
  uint32_t after_bound = (bound << 1) | (L.pb == L.p0 - 1 ? 1u : 0u);
  if (L.p0 < 0 && L.p0 + 16 > 0) after_bound |= 1u << (-L.p0);  // offset 0 behaves like "just after a boundary"
  L.ne = delims & ~after_bound;
  // counts in front of the lane: one packed inclusive scan (each count <= 16 per lane, <= 512 per step)
  const uint32_t mine = (uint32_t)__popc(L.term) | ((uint32_t)__popc(L.tab) << 10) | ((uint32_t)__popc(L.ne) << 20);
  uint32_t inc = mine;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= (unsigned)o) inc += t;
  }
  const uint32_t ex = inc - mine;
  L.rows = c.rows + (ex & 1023u);
  L.tabs = c.tabs + ((ex >> 10) & 1023u);
  L.nes = c.ne + (ex >> 20);
  const uint32_t tot = __shfl_sync(0xffffffffu, inc, 31);
  c.rows += tot & 1023u;
  c.tabs += (tot >> 10) & 1023u;
  c.ne += tot >> 20;
  return L;
}

// ---------------------------------------------------------------------------------------------
// census: counts per tile
// ---------------------------------------------------------------------------------------------
// The census needs totals only, so it runs a lighter version of scan_step: the same masks, but counts are summed per
// lane and reduced once per tile, and "the byte in front is a boundary" travels as one bit instead of a position.
__global__ void __launch_bounds__(ENC_THREADS)
    k_tile_count(const uint8_t* __restrict__ buf, uint64_t n, int64_t lo, uint32_t ntiles, TileAgg* __restrict__ agg) {
  const uint32_t tile = blockIdx.x * ENC_WARPS + (threadIdx.x >> 5);
  if (tile >= ntiles) return;
  const unsigned lane = lane_id();
  const int64_t t0 = lo + (int64_t)tile * TILE, limit = (int64_t)n;
  uint32_t c_bs = (t0 > 0 && __ldg(buf + t0 - 1) == (uint8_t)'\\') ? 1u : 0u;
  uint32_t c_nl = t0 <= 0 ? 1u : (is_unescaped_newline(buf, t0 - 1) ? 1u : 0u);
  uint32_t c_bd = t0 == 0 ? 1u : 0u;  // the byte in front of the tile is a boundary (buffer start counts as one)
  if (t0 > 0) {
    const uint8_t b = __ldg(buf + t0 - 1);
    if ((b == (uint8_t)'\t' || b == (uint8_t)'\n') && !odd_backslashes_before(buf, t0 - 1)) c_bd = 1u;
  }
  uint32_t rows = 0, tabs = 0, ne = 0;
  int32_t last_b = -1, last_r = -1;  // offsets inside the tile
  for (uint32_t s = 0; s < TILE; s += STEP) {
    const int64_t p0 = t0 + s + 16 * (int64_t)lane;
    uint32_t tab = 0, nl = 0, bs = 0;
    if (p0 < limit && p0 + 16 > 0) {
      const uint4 v = ldg_stream_u4(buf + p0);
      const int64_t ia = p0 < 0 ? -p0 : 0;
      const int64_t ib = p0 + 16 > limit ? limit - p0 : 16;
      const uint32_t in = ((1u << ib) - 1u) & ~((1u << ia) - 1u);
      tab = chunk_mask(v, '\t') & in;
      if (chunk_has(v, '\n')) nl = chunk_mask(v, '\n') & in;
      if (chunk_has(v, '\\')) bs = chunk_mask(v, '\\') & in;
    }
    uint32_t prev = __shfl_up_sync(0xffffffffu, bs >> 15, 1);
    if (lane == 0) prev = c_bs;
    uint32_t sus = (tab | nl) & ((bs << 1) | prev);
    while (sus) {  // escape parity: only delimiters that directly follow a backslash need the (rare) backward walk
      const int i = __ffs(sus) - 1;
      sus &= sus - 1;
      if (odd_backslashes_before(buf, p0 + i)) {
        tab &= ~(1u << i);
        nl &= ~(1u << i);
      }
    }
    uint32_t prevnl = __shfl_up_sync(0xffffffffu, nl >> 15, 1);
    if (lane == 0) prevnl = c_nl;
    uint32_t after_nl = ((nl << 1) | prevnl) & 0xffffu;
    const bool has_zero = p0 <= 0 && p0 + 16 > 0;
    if (has_zero) after_nl |= 1u << (-p0);
    const uint32_t skip = nl & after_nl, term = nl & ~skip, bound = tab | nl;
    uint32_t prevbd = __shfl_up_sync(0xffffffffu, bound >> 15, 1);
    if (lane == 0) prevbd = c_bd;
    uint32_t after_bound = (bound << 1) | prevbd;
    if (has_zero) after_bound |= 1u << (-p0);
    rows += (uint32_t)__popc(term);
    tabs += (uint32_t)__popc(tab);
    ne += (uint32_t)__popc((tab | term) & ~after_bound);
    if (bound) last_b = (int32_t)(s + 16u * lane) + (31 - __clz(bound));
    if (nl) last_r = (int32_t)(s + 16u * lane) + (31 - __clz(nl));
    c_bs = __shfl_sync(0xffffffffu, bs >> 15, 31);
    c_nl = __shfl_sync(0xffffffffu, nl >> 15, 31);
    c_bd = __shfl_sync(0xffffffffu, bound >> 15, 31);
  }
  rows = __reduce_add_sync(0xffffffffu, rows);
  tabs = __reduce_add_sync(0xffffffffu, tabs);
  ne = __reduce_add_sync(0xffffffffu, ne);
  last_b = __reduce_max_sync(0xffffffffu, last_b);
  last_r = __reduce_max_sync(0xffffffffu, last_r);
  if (lane == 0) {
    TileAgg a;
    a.rows = rows;
    a.tabs = tabs;
    a.ne = ne;
    a.bound_p1 = last_b >= 0 ? (uint32_t)(t0 + last_b + 1) : 0u;
    a.break_p1 = last_r >= 0 ? (uint32_t)(t0 + last_r + 1) : 0u;
    a.rs_p1 = 0u;
    agg[tile] = a;
  }
}

// single CTA: exclusive prefix of the tile aggregates (sums for the counts, running maximum for the positions)
constexpr int TS_THREADS = 1024;
__device__ __forceinline__ TileAgg agg_join(const TileAgg& a, const TileAgg& b) {
  TileAgg r;
  r.rows = a.rows + b.rows;
  r.tabs = a.tabs + b.tabs;
  r.ne = a.ne + b.ne;
  r.bound_p1 = max(a.bound_p1, b.bound_p1);
  r.break_p1 = max(a.break_p1, b.break_p1);
  r.rs_p1 = max(a.rs_p1, b.rs_p1);
  return r;
}
__device__ __forceinline__ TileAgg agg_shfl_up(const TileAgg& a, int o) {
  TileAgg r;
  r.rows = __shfl_up_sync(0xffffffffu, a.rows, o);
  r.tabs = __shfl_up_sync(0xffffffffu, a.tabs, o);
  r.ne = __shfl_up_sync(0xffffffffu, a.ne, o);
  r.bound_p1 = __shfl_up_sync(0xffffffffu, a.bound_p1, o);
  r.break_p1 = __shfl_up_sync(0xffffffffu, a.break_p1, o);
  r.rs_p1 = __shfl_up_sync(0xffffffffu, a.rs_p1, o);
  return r;
}
__global__ void __launch_bounds__(TS_THREADS) k_tile_scan(TileAgg* __restrict__ agg, uint32_t ntiles, EncMeta* __restrict__ meta) {
  __shared__ TileAgg wsum[32];
  const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const TileAgg zero = {0u, 0u, 0u, 0u, 0u, 0u};
  TileAgg carry = zero;  // everything in front of the current round of 1024 tiles
  for (uint32_t base = 0; base < ntiles; base += TS_THREADS) {
    const uint32_t t = base + threadIdx.x;
    const TileAgg mine = t < ntiles ? agg[t] : zero;
    TileAgg inc = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const TileAgg u = agg_shfl_up(inc, o);
      if (lane >= (unsigned)o) inc = agg_join(u, inc);
    }
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    if (warp == 0) {
      TileAgg w = wsum[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const TileAgg u = agg_shfl_up(w, o);
        if (lane >= (unsigned)o) w = agg_join(u, w);
      }
      wsum[lane] = w;  // inclusive over warps
    }
    __syncthreads();
    TileAgg ex = carry;
    if (warp) ex = agg_join(ex, wsum[warp - 1]);
    const TileAgg up = agg_shfl_up(inc, 1);
    if (lane) ex = agg_join(ex, up);
    if (t < ntiles) agg[t] = ex;
    carry = agg_join(carry, wsum[31]);
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    meta->tot_rows = carry.rows;
    meta->tot_tabs = carry.tabs;
    meta->tot_ne = carry.ne;
    meta->last_break_p1 = carry.break_p1;
  }
}

// The same prefix over many CTAs: every CTA scans 1024 tiles in place and reports its total; k_tile_scan then runs over
// the CTA totals (and fills in the census totals), k_tile_scan_add folds them back in.
__global__ void __launch_bounds__(TS_THREADS) k_tile_scan_local(TileAgg* __restrict__ agg, uint32_t ntiles, TileAgg* __restrict__ part) {
  __shared__ TileAgg wsum[32];
  const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const TileAgg zero = {0u, 0u, 0u, 0u, 0u, 0u};
  const uint32_t t = blockIdx.x * TS_THREADS + threadIdx.x;
  const TileAgg mine = t < ntiles ? agg[t] : zero;
  TileAgg inc = mine;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const TileAgg u = agg_shfl_up(inc, o);
    if (lane >= (unsigned)o) inc = agg_join(u, inc);
  }
  if (lane == 31) wsum[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    TileAgg w = wsum[lane];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const TileAgg u = agg_shfl_up(w, o);
      if (lane >= (unsigned)o) w = agg_join(u, w);
    }
    wsum[lane] = w;  // inclusive over warps
  }
  __syncthreads();
  TileAgg ex = zero;
  if (warp) ex = wsum[warp - 1];
  const TileAgg up = agg_shfl_up(inc, 1);
  if (lane) ex = agg_join(ex, up);
  if (t < ntiles) agg[t] = ex;
  if (threadIdx.x == 0) part[blockIdx.x] = wsum[31];
}
__global__ void __launch_bounds__(TS_THREADS) k_tile_scan_add(TileAgg* __restrict__ agg, uint32_t ntiles, const TileAgg* __restrict__ part) {
  const uint32_t t = blockIdx.x * TS_THREADS + threadIdx.x;
  if (t < ntiles && blockIdx.x) agg[t] = agg_join(part[blockIdx.x], agg[t]);
}

// one warp: terminator of row `want` (0-based) -> meta->cut_end_p1, first byte of the next row -> meta->next_start
__global__ void k_find_cut(const uint8_t* __restrict__ buf, uint64_t n, int64_t lo, uint32_t ntiles, uint32_t tile_bytes,
                           const TileAgg* __restrict__ pre, uint32_t want, EncMeta* __restrict__ meta) {
  // largest tile whose exclusive row prefix is <= want
  uint32_t a = 0, b = ntiles;
  while (b - a > 1) {
    const uint32_t m = (a + b) >> 1;
    if (pre[m].rows <= want) a = m;
    else b = m;
  }
  const int64_t t0 = lo + (int64_t)a * tile_bytes;
  WarpCarry c;
  carry_init(buf, t0, pre[a], c);
  for (uint32_t s = 0; s < tile_bytes; s += STEP) {
    const LaneStep L = scan_step(buf, (int64_t)n, t0 + s, c);
    uint32_t t = L.term;
    while (t) {
      const int i = __ffs(t) - 1;
      t &= t - 1;
      if (L.rows + (uint32_t)__popc(L.term & ((1u << i) - 1u)) == want) {
        const uint64_t pos = (uint64_t)(L.p0 + i);
        uint64_t nx = pos + 1;
        while (nx < n && __ldg(buf + nx) == (uint8_t)'\n') ++nx;  // blank lines directly after a row are skipped
        meta->cut_end_p1 = (uint32_t)(pos + 1);
        meta->next_start = (uint32_t)nx;
      }
    }
  }
}

// The row after the block's last one (the reference's interrupted row, SURVEY App. B-14): one thread walks it from
// `start` with the delimiter rules of scan_step and reports where its first `spill_cols` columns end and how long it is.
__global__ void k_find_spill(const uint8_t* __restrict__ buf, uint64_t n, uint32_t start, uint32_t spill_cols,
                             EncMeta* __restrict__ meta) {
  uint32_t closed = 0, spill_end = start, odd = 0;
  uint32_t row_len = 0;
  for (uint64_t p = start; p < n; ++p) {
    const uint8_t b = buf[p];
    if (b == (uint8_t)'\\') {
      odd ^= 1u;
      continue;
    }
    const bool escaped = odd != 0u;
    odd = 0;
    if (escaped) continue;
    if (b == (uint8_t)'\t' || b == (uint8_t)'\n') {
      if (closed < spill_cols) {
        ++closed;
        spill_end = (uint32_t)p + 1u;
      }
      if (b == (uint8_t)'\n') {
        row_len = (uint32_t)(p - start) + 1u;
        break;
      }
    }
  }
  meta->spill_end = row_len ? spill_end : start;  // an unterminated tail is not a row: nothing spills
  meta->spill_row_len = row_len;
}

// ---------------------------------------------------------------------------------------------
// string hash set (open addressing, 64-bit slots: (start+1) << 32 | len, 0 = empty)
// ---------------------------------------------------------------------------------------------
struct HashTable {
  unsigned long long* slots;
  uint32_t mask;
};

__device__ __forceinline__ uint32_t rotl32(uint32_t x, int r) { return __funnelshift_l(x, x, r); }

// The hash is a SUM of position-keyed word mixes, so one lane can evaluate it straight-line for short strings and a
// group of lanes can evaluate it cooperatively for long ones, with the same result.
__device__ __forceinline__ uint32_t mix_word(uint32_t w, uint32_t i) {
  uint32_t x = w ^ (i * 0x9E3779B1u + 0x85EBCA77u);
  x *= 0xCC9E2D51u;
  x = rotl32(x, 15);
  x *= 0x1B873593u;
  return x;
}
__device__ __forceinline__ uint32_t finish_hash(uint32_t sum, uint32_t len) {
  uint32_t h = sum ^ (len * 0x27D4EB2Fu);
  h ^= h >> 16;
  h *= 0x85EBCA6Bu;
  h ^= h >> 13;
  h *= 0xC2B2AE35u;
  h ^= h >> 16;
  return h;
}

// Little-endian word k (bytes 4k .. 4k+3, zero beyond len) of the string at s; `wlast` = last readable aligned word.
struct StrWords {
  const uint32_t* w;
  uint32_t sh;
  const uint32_t* wlast;
  __device__ __forceinline__ StrWords(const uint8_t* s, const uint32_t* last) : wlast(last) {
    const uintptr_t a = reinterpret_cast<uintptr_t>(s);
    w = reinterpret_cast<const uint32_t*>(a & ~(uintptr_t)3);
    sh = (uint32_t)(a & 3u) * 8u;
  }
  __device__ __forceinline__ uint32_t word(uint32_t k, uint32_t len) const {
    const uint32_t* p = w + k;
    const uint32_t a = __ldg(p);
    const uint32_t b = sh ? __ldg(p + 1 <= wlast ? p + 1 : wlast) : 0u;
    const uint32_t x = __funnelshift_r(a, b, sh);
    const uint32_t rem = len - 4u * k;
    return rem >= 4u ? x : (x & ((1u << (8u * rem)) - 1u));
  }
};

// short strings: the first NW masked words (NW = 4 covers 16 bytes, NW = 5 the 19 digits of a 64-bit number)
template <int NW>
__device__ __forceinline__ void short_words(const uint8_t* s, uint32_t len, const uint32_t* wlast, uint32_t x[NW]) {
  const uintptr_t a = reinterpret_cast<uintptr_t>(s);
  const uint32_t* w = reinterpret_cast<const uint32_t*>(a & ~(uintptr_t)3);
  const uint32_t sh = (uint32_t)(a & 3u) * 8u;
  const uint32_t room = (uint32_t)min((ptrdiff_t)NW, wlast - w);
  uint32_t prev = __ldg(w);
#pragma unroll
  for (uint32_t k = 0; k < NW; ++k) {
    const uint32_t nx = __ldg(w + min(k + 1u, room));
    x[k] = __funnelshift_r(prev, nx, sh);
    prev = nx;
  }
#pragma unroll
  for (uint32_t k = 0; k < NW; ++k) {
    const uint32_t got = len > 4u * k ? len - 4u * k : 0u;
    x[k] = got >= 4u ? x[k] : (got ? (x[k] & ((1u << (8u * got)) - 1u)) : 0u);
  }
}
// ---------------------------------------------------------------------------------------------
// pass 1
// ---------------------------------------------------------------------------------------------
struct P1Args {
  const uint8_t* buf;
  uint64_t n;          // readable bytes
  int64_t lo;          // -(buf & 15)
  int64_t limit;       // bytes of the block: delimiters at or beyond it are not part of it
  uint32_t ntiles, ncols;
  const TileAgg* pre;
  const uint8_t* types;
  int trim;
  HashTable ht;
  uint32_t* colset;
  unsigned long long* colmin;
  unsigned long long* colmax;
  uint32_t* rec_col;             // [tot_ne]
  unsigned long long* rec_val;   // [tot_ne] dictionary slot (text) or pass-2 number
  uint32_t* row_rec;             // [rows + 1] records in front of row r
  EncMeta* meta;
};

constexpr uint32_t QN = 320;  // fields a warp can hold: up to 31 left over + the 256 a step can produce, rounded up

struct P1Warp {        // per-warp shared memory: non-empty fields in row order, not yet processed
  uint32_t start[QN], len[QN], col[QN];
};

struct P1Stats {
  uint32_t new_count, max_len, max_line;
  unsigned long long new_bytes;
};

// 8 lanes (one octet of the warp) work on one long string: gl = lane within the octet, `om` = the octet's lane mask.
__device__ __forceinline__ uint32_t ht_upsert_long(const P1Args& A, const uint32_t* wlast, uint32_t start, uint32_t len, unsigned gl,
                                                   unsigned om, bool active, bool* is_new) {
  *is_new = false;
  const uint32_t nw = (len + 3u) >> 2;
  uint32_t s = 0;
  if (active) {
    const StrWords me(A.buf + start, wlast);
    for (uint32_t k = gl; k < nw; k += 8) s += mix_word(me.word(k, len), k);
  }
  s += __shfl_xor_sync(0xffffffffu, s, 1);
  s += __shfl_xor_sync(0xffffffffu, s, 2);
  s += __shfl_xor_sync(0xffffffffu, s, 4);
  uint32_t i = finish_hash(s, len) & A.ht.mask;
  const unsigned long long mine = ((unsigned long long)(start + 1u) << 32) | len;
  uint32_t result = 0;
  bool done = !active;
  for (uint32_t probe = 0; probe < HT_MAX_PROBE; ++probe) {
    // every octet runs the same number of iterations (the shuffles below are warp-wide)
    unsigned long long cur = 0;
    if (!done) {
      cur = A.ht.slots[i];
      if (cur == 0ull) {
        if (gl == 0) cur = atomicCAS(&A.ht.slots[i], 0ull, mine);
      }
    }
    // lane 0 of the octet decides
    const unsigned long long cur0 = __shfl_sync(0xffffffffu, cur, (lane_id() & ~7u));
    bool match = false;
    if (!done) {
      if (cur0 == 0ull) {  // our CAS went through
        *is_new = true;
        result = i;
        done = true;
      } else if ((uint32_t)cur0 == len) {
        const uint32_t cs = (uint32_t)(cur0 >> 32) - 1u;
        match = true;
        if (cs != start) {
          const StrWords me(A.buf + start, wlast), other(A.buf + cs, wlast);
          for (uint32_t k = gl; k < nw && match; k += 8) match = me.word(k, len) == other.word(k, len);
        }
      }
    }
    const unsigned votes = __ballot_sync(0xffffffffu, match || done);
    if (!done) {
      if ((votes & om) == om && (uint32_t)cur0 == len && cur0 != 0ull) {
        result = i;
        done = true;
      } else {
        i = (i + 1) & A.ht.mask;
      }
    }
    if (__all_sync(0xffffffffu, done)) return result;
  }
  if (!done) *reinterpret_cast<volatile uint32_t*>(&A.meta->ht_overflow) = 1u;
  return result;
}

__device__ __forceinline__ uint32_t trimmed_len(const uint8_t* __restrict__ buf, uint32_t start, uint32_t len) {
  while (len && __ldg(buf + start + len - 1) == (uint8_t)' ') --len;  // -t: ConvertToZDW.cpp:295-313
  return len;
}

// ---------------------------------------------------------------------------------------------
// Field processing.  The warp's main queue holds every non-empty field in row order (slot = ordinal).  In a batch of
// 32, everything that fits 20 bytes - numbers, CHAR cells and texts of up to SHORT_MAX bytes, the bulk of
// analytics-shaped data - is served from five register words loaded once; texts of SHORT_MAX+1 .. MID_MAX bytes are
// parked in a small per-warp ring and worked off 32 at a time, one lane each; the rare longer texts are handled in
// place by the octets of the warp.
// ---------------------------------------------------------------------------------------------
constexpr uint32_t MID_MAX = 128;  // longest text handled by a single lane (measured: 32 -> 1.66, 64 -> 1.53, 128 -> 1.51 ms)
constexpr uint32_t SQ = 64;        // entries of a side queue (at most 31 waiting + 32 pushed)

struct P1Side {  // a ring; `end` = entries ever pushed, `done` = entries ever taken (warp-uniform, kept here)
  uint32_t start[SQ], len[SQ], col[SQ], ord[SQ];
  uint32_t end, done;
};

// all lanes call; returns the number of entries waiting afterwards
__device__ __forceinline__ uint32_t side_push(P1Side& Q, bool want, uint32_t start, uint32_t len, uint32_t col, uint32_t ord) {
  const unsigned m = __ballot_sync(0xffffffffu, want);
  const uint32_t end = Q.end;
  if (want) {
    const uint32_t i = (end + (uint32_t)__popc(m & lanemask_lt())) & (SQ - 1u);
    Q.start[i] = start;
    Q.len[i] = len;
    Q.col[i] = col;
    Q.ord[i] = ord;
  }
  __syncwarp();
  const uint32_t e2 = end + (uint32_t)__popc(m);
  if (m && lane_id() == 0) Q.end = e2;
  return e2 - Q.done;
}

__device__ __forceinline__ void note_new_string(P1Stats& st, uint32_t len) {
  ++st.new_count;
  st.new_bytes += (unsigned long long)len + 1ull;
  st.max_len = max(st.max_len, len);
}

// Column statistics.  The loads that filter the atomics may come from a stale L1 line: the three arrays only move one
// way (set 0 -> 1, min down, max up), so a stale value can cost a redundant atomic but never skips a needed one.
#define P1_LD(p) (*(p))
__device__ __forceinline__ void note_column_set(const P1Args& A, uint32_t col) {
  if (P1_LD(A.colset + col) == 0u) A.colset[col] = 1u;
}
__device__ __forceinline__ void note_column_value(const P1Args& A, uint32_t col, unsigned long long v1) {
  if (v1 != 0) {  // zero / empty numeric cells take no part in min/max: ConvertToZDW.cpp:362,386
    note_column_set(A, col);
    if (v1 < P1_LD(A.colmin + col)) atomicMin(A.colmin + col, v1);
    if (v1 > P1_LD(A.colmax + col)) atomicMax(A.colmax + col, v1);
  }
}

// one text, any length, by a single lane: words streamed four at a time through a funnel shift.  The record's value is
// the string's hash-set slot + BIAS (the delta path uses BIAS = 1 so that 0 can mean "the field became empty")
template <uint32_t BIAS = 0>
__device__ __forceinline__ void text_one(const P1Args& A, const uint32_t* wlast, uint32_t start, uint32_t len, uint32_t col,
                                            uint32_t ord, P1Stats& st) {
  const uint32_t nw = (len + 3u) >> 2;
  const uint32_t tail = len & 3u, tail_mask = tail ? ((1u << (8u * tail)) - 1u) : 0xffffffffu;
  const uintptr_t a = reinterpret_cast<uintptr_t>(A.buf + start);
  const uint32_t* w = reinterpret_cast<const uint32_t*>(a & ~(uintptr_t)3);
  const uint32_t sh = (uint32_t)(a & 3u) * 8u;
  const uint32_t room = (uint32_t)min((ptrdiff_t)0x7fffffff, wlast - w);  // whole words readable after *w
  uint32_t sum = 0;
  {
    uint32_t prev = __ldg(w);
    for (uint32_t k0 = 0; k0 < nw; k0 += 4u) {
      const uint32_t n0 = __ldg(w + min(k0 + 1u, room)), n1 = __ldg(w + min(k0 + 2u, room)), n2 = __ldg(w + min(k0 + 3u, room)),
                     n3 = __ldg(w + min(k0 + 4u, room));
      uint32_t x0 = __funnelshift_r(prev, n0, sh), x1 = __funnelshift_r(n0, n1, sh), x2 = __funnelshift_r(n1, n2, sh),
               x3 = __funnelshift_r(n2, n3, sh);
      prev = n3;
      const uint32_t left = nw - k0;  // words of the text in this group (>= 1)
      if (left == 1u) x0 &= tail_mask;
      if (left == 2u) x1 &= tail_mask;
      if (left == 3u) x2 &= tail_mask;
      if (left == 4u) x3 &= tail_mask;
      sum += mix_word(x0, k0);
      if (left > 1u) sum += mix_word(x1, k0 + 1u);
      if (left > 2u) sum += mix_word(x2, k0 + 2u);
      if (left > 3u) sum += mix_word(x3, k0 + 3u);
    }
  }
  uint32_t i = finish_hash(sum, len) & A.ht.mask;
  const unsigned long long mine = ((unsigned long long)(start + 1u) << 32) | len;
  bool is_new = false, found = false;
  for (uint32_t probe = 0; probe < HT_MAX_PROBE; ++probe) {
    unsigned long long cur = A.ht.slots[i];
    if (cur == 0ull) {
      cur = atomicCAS(&A.ht.slots[i], 0ull, mine);
      if (cur == 0ull) {
        is_new = true;
        found = true;
        break;
      }
    }
    if ((uint32_t)cur == len) {
      const uint32_t cs = (uint32_t)(cur >> 32) - 1u;
      uint32_t diff = 0;
      if (cs != start) {
        const uintptr_t b = reinterpret_cast<uintptr_t>(A.buf + cs);
        const uint32_t* v = reinterpret_cast<const uint32_t*>(b & ~(uintptr_t)3);
        const uint32_t sh2 = (uint32_t)(b & 3u) * 8u;
        const uint32_t room2 = (uint32_t)min((ptrdiff_t)0x7fffffff, wlast - v);
        uint32_t p1 = __ldg(w), p2 = __ldg(v);
        for (uint32_t k0 = 0; k0 < nw && diff == 0u; k0 += 4u) {
          const uint32_t a0 = __ldg(w + min(k0 + 1u, room)), a1 = __ldg(w + min(k0 + 2u, room)), a2 = __ldg(w + min(k0 + 3u, room)),
                         a3 = __ldg(w + min(k0 + 4u, room));
          const uint32_t b0 = __ldg(v + min(k0 + 1u, room2)), b1 = __ldg(v + min(k0 + 2u, room2)),
                         b2 = __ldg(v + min(k0 + 3u, room2)), b3 = __ldg(v + min(k0 + 4u, room2));
          uint32_t d0 = __funnelshift_r(p1, a0, sh) ^ __funnelshift_r(p2, b0, sh2);
          uint32_t d1 = __funnelshift_r(a0, a1, sh) ^ __funnelshift_r(b0, b1, sh2);
          uint32_t d2 = __funnelshift_r(a1, a2, sh) ^ __funnelshift_r(b1, b2, sh2);
          uint32_t d3 = __funnelshift_r(a2, a3, sh) ^ __funnelshift_r(b2, b3, sh2);
          p1 = a3;
          p2 = b3;
          const uint32_t left = nw - k0;
          if (left == 1u) d0 &= tail_mask;
          if (left == 2u) d1 &= tail_mask;
          if (left == 3u) d2 &= tail_mask;
          if (left == 4u) d3 &= tail_mask;
          diff = d0 | (left > 1u ? d1 : 0u) | (left > 2u ? d2 : 0u) | (left > 3u ? d3 : 0u);
        }
      }
      if (diff == 0u) {
        found = true;
        break;
      }
    }
    i = (i + 1) & A.ht.mask;
  }
  if (!found) {
    *reinterpret_cast<volatile uint32_t*>(&A.meta->ht_overflow) = 1u;
    i = 0;
  }
  A.rec_col[ord] = col;
  A.rec_val[ord] = (unsigned long long)i + BIAS;
  note_column_set(A, col);
  if (is_new) note_new_string(st, len);
}

// Processes the queued fields [off, off + count) of the warp's main queue (count <= 32): lane l takes field off + l.
// Q[0] parks texts of up to SHORT_MAX bytes, Q[1] texts of up to MID_MAX bytes; longer ones go to the octets at once.
// QT = the queue's arrays (start / len / col); `ords` (may be null) = the record every field fills, else ord0 + lane.
// BIAS is added to the hash-set slot a text's record holds (the delta path keeps 0 for "became empty").
template <uint32_t BIAS, class QT>
__device__ __forceinline__ void p1_process(const P1Args& A, const uint32_t* wlast, const QT& W, uint32_t off, uint32_t count,
                                           uint32_t ord0, const uint32_t* ords, P1Stats& st, P1Side* Q, bool flush) {
  const unsigned lane = lane_id();
  const bool valid = lane < count;
  uint32_t start = 0, len = 0, col = 0;
  uint8_t t = 0;
  if (valid) {
    start = W.start[off + lane];
    len = W.len[off + lane];
    col = W.col[off + lane];
    t = __ldg(A.types + col);
  }
  const uint32_t ord = ords ? (valid ? ords[off + lane] : 0u) : ord0 + lane;
  const uint32_t ord_src = ord;  // (long texts below fetch the source lane's record by shuffle)
  const bool live = valid && len != 0u;
  const bool text = is_text_like(t);
  if (BIAS == 0u && valid && len == 0u) A.rec_col[ord] = REC_EMPTY;  // -t turned the field into an empty one (or the row is malformed)
  // The row-delta path (BIAS 1) also takes the "became empty" records (len 0), and parses the field the column had in
  // the row before as well - k_pass1d left its place in rec_val - so that the record can say whether the value changed
  if (!text && (BIAS == 0u ? live : valid)) {
    unsigned long long v1 = 0, v2 = 0, old = 0;
    const unsigned long long prev = BIAS ? A.rec_val[ord] : 0ull;
#pragma unroll 1
    for (uint32_t h = 0; h < (BIAS ? 2u : 1u); ++h) {
      const uint32_t fs = h ? (uint32_t)(prev >> 32) : start, fl = h ? (uint32_t)prev : len;
      unsigned long long a = 0, b = 0;
      if (fl && (fl <= NUM_FAST_MAX || t == ZDWB_CHAR)) {
        uint32_t x[5];
        short_words<5>(A.buf + fs, fl, wlast, x);
        if (t == ZDWB_CHAR) {
          // sign-extended first byte (+ second byte * 256): min/max rule ConvertToZDW.cpp:358-361 (second byte only
          // after a backslash), pass-2 rule :543-547 (always); bytes past the field read as NUL (x is masked)
          const long long b0 = (long long)(int8_t)(x[0] & 0xffu);
          const long long b1 = fl > 1 ? (long long)((int32_t)(int8_t)((x[0] >> 8) & 0xffu) * 256) : 0ll;
          a = (unsigned long long)(b0 + ((x[0] & 0xffu) == (uint32_t)'\\' ? b1 : 0ll));
          b = (unsigned long long)(b0 + b1);
        } else {
          // strtoull (:385,564): an optional sign in front of the digits ('-' negates modulo 2^64; with a sign at most
          // 19 digits are left, which cannot overflow); anything else - white space, junk - takes the exact byte walk
          if (!fast_number(x, fl, &a)) a = parse_u64_field(A.buf + fs, fl);
          b = a;
        }
      } else if (fl) {  // a number of more than 20 characters
        a = b = parse_u64_field(A.buf + fs, fl);
      }
      if (h) {
        old = b;
      } else {
        v1 = a;
        v2 = b;
      }
    }
    // (pass 2's flag is mapped(v2) != mapped(old), mapped(v) = v ? v - base : 0.  That is v2 != old: subtracting the
    // base is injective, and a non-zero v2 never equals the base - DESIGN 3 shows it for CHAR cells too)
    A.rec_col[ord] = BIAS && v2 == old ? col | REC_SAME : col;
    A.rec_val[ord] = v2;
    note_column_value(A, col, v1);
  }
  if (BIAS != 0u && valid && text && len == 0u) A.rec_val[ord] = 0ull;  // a text column became empty: value 0, flag set
  const bool is_text = live && text;
  uint32_t waiting[2];
  waiting[0] = side_push(Q[0], is_text && len <= SHORT_MAX, start, len, col, ord);
  waiting[1] = side_push(Q[1], is_text && len > SHORT_MAX && len <= MID_MAX, start, len, col, ord);
  // ---- long texts: octet g takes the g-th, (g+4)-th, ... of them
  unsigned todo = __ballot_sync(0xffffffffu, is_text && len > MID_MAX);
  if (todo) {
    const unsigned grp = lane >> 3, gl = lane & 7u, om = 0xffu << (grp * 8);
    while (todo) {
      // the source lane of this octet: the (grp+1)-th set bit of todo
      unsigned m = todo;
      for (unsigned k = 0; k < grp && m; ++k) m &= m - 1;
      const bool active = m != 0u;
      const int src = active ? __ffs(m) - 1 : 0;
      const uint32_t s2 = __shfl_sync(0xffffffffu, start, src), l2 = __shfl_sync(0xffffffffu, len, src),
                     c2 = __shfl_sync(0xffffffffu, col, src);
      bool is_new;
      const uint32_t slot = ht_upsert_long(A, wlast, s2, l2, gl, om, active, &is_new);
      const uint32_t o2 = __shfl_sync(0xffffffffu, ord_src, src);
      if (active && gl == 0) {
        A.rec_col[o2] = c2;
        A.rec_val[o2] = (unsigned long long)slot + BIAS;
        note_column_set(A, c2);
        if (is_new) note_new_string(st, l2);
      }
      // drop the (up to) four texts just handled
      for (int k = 0; k < 4 && todo; ++k) todo &= todo - 1;
    }
  }
  // ---- parked texts, 32 of a kind at a time (one call site: the loop is not unrolled)
#pragma unroll 1
  for (uint32_t qi = 0; qi < 2u; ++qi) {
    uint32_t n = qi ? waiting[1] : waiting[0];
    while (n >= 32u || (flush && n)) {
      P1Side& S = Q[qi];
      const uint32_t take = min(n, 32u), head = S.done;
      if (lane < take) {
        const uint32_t e = (head + lane) & (SQ - 1u);
        text_one<BIAS>(A, wlast, S.start[e], S.len[e], S.col[e], S.ord[e], st);
      }
      __syncwarp();
      if (lane == 0) S.done = head + take;
      __syncwarp();
      n -= take;
    }
  }
}

__global__ void __launch_bounds__(ENC_THREADS, 4) k_pass1(const P1Args A) {
  __shared__ P1Warp sw[ENC_WARPS];
  __shared__ P1Side s_side[ENC_WARPS][2];
  const unsigned lane = lane_id(), warp = threadIdx.x >> 5;
  const uint32_t tile = blockIdx.x * ENC_WARPS + warp;
  if (tile >= A.ntiles) return;
  P1Warp& W = sw[warp];
  const int64_t t0 = A.lo + (int64_t)tile * TILE;
  if (t0 >= A.limit) return;
  const uint32_t* wlast = reinterpret_cast<const uint32_t*>(reinterpret_cast<uintptr_t>(A.buf + A.n - 1) & ~(uintptr_t)3);
  WarpCarry c;
  carry_init(A.buf, t0, A.pre[tile], c);
  P1Stats st = {0u, 0u, 0u, 0ull};
  P1Side* Q = s_side[warp];
  if (lane < 2) Q[lane].end = Q[lane].done = 0u;
  __syncwarp();
  uint32_t qbase = c.ne;  // ordinal of the field held in queue slot 0
  const uint32_t tabs_per_row = A.ncols - 1u;
  if (tile == 0 && lane == 0) A.row_rec[0] = 0u;

  // One call site for the field processing keeps the kernel small (it is instruction-cache sensitive): the loop runs
  // one extra round after the last step, in which the leftover fields and the side queue are flushed.
  for (uint32_t s = 0;; s += STEP) {
    const bool last = s >= TILE || t0 + (int64_t)s >= A.limit;
    if (!last) {
      const uint32_t ne_before = c.ne;
      const LaneStep L = scan_step(A.buf, A.limit, t0 + s, c);
      // ---- rows that end here: field-count check, longest line, record index of the next row
      uint32_t tm = L.term;
      while (tm) {
        const int i = __ffs(tm) - 1;
        tm &= tm - 1;
        const uint32_t below = (1u << i) - 1u;
        const uint32_t R = L.rows + (uint32_t)__popc(L.term & below);
        const uint32_t T = L.tabs + (uint32_t)__popc(L.tab & below);
        if (T != (R + 1u) * tabs_per_row) atomicMin(&A.meta->bad_row, R);  // cumulative: exact for the first bad row
        const uint32_t brk = (L.term | L.skip) & below;
        const int64_t row_start = (brk ? L.p0 + (31 - __clz(brk)) : L.prb) + 1;
        st.max_line = max(st.max_line, (uint32_t)(L.p0 + i - row_start + 1));
        A.row_rec[R + 1u] = L.nes + (uint32_t)__popc(L.ne & ((2u << i) - 1u));
      }
      // ---- non-empty fields go to the warp's queue, slot = ordinal.  Two phases, so that a lane that scanned a run of
      // short fields does not hold up the warp: every lane first drops the bit position (lane * 16 + bit) of each of
      // its closing delimiters into the field's slot; then the step's fields are dealt out evenly, field k to lane
      // k & 31, which fetches the scanning lane's masks by shuffle and works out column, start and length.
      {
        uint32_t rem = L.ne, q = L.nes - qbase;
        while (rem) {
          W.start[q++] = lane * 16u + (uint32_t)(__ffs(rem) - 1);
          rem &= rem - 1;
        }
      }
      __syncwarp();
      {
        const uint32_t nf = c.ne - ne_before, qb = ne_before - qbase;
        const uint32_t pk_tt = L.tab | (L.term << 16), pk_bd = L.tab | L.term | L.skip;
        const uint32_t colbase = L.tabs - L.rows * tabs_per_row;
        for (uint32_t k0 = 0; k0 < nf; k0 += 32u) {
          const uint32_t k = k0 + lane;
          const bool mine = k < nf;
          const uint32_t pos = mine ? W.start[qb + k] : 0u;
          const int j = (int)(pos >> 4);
          const uint32_t i = pos & 15u;
          const uint32_t tt = __shfl_sync(0xffffffffu, pk_tt, j), bd = __shfl_sync(0xffffffffu, pk_bd, j);
          const uint32_t cb = __shfl_sync(0xffffffffu, colbase, j);
          const int64_t pb_j = __shfl_sync(0xffffffffu, L.pb, j);
          if (mine) {
            const uint32_t below = (1u << i) - 1u;
            const int64_t p0 = t0 + (int64_t)s + 16 * (int64_t)j;
            uint32_t col = cb + (uint32_t)__popc(tt & below) - (uint32_t)__popc((tt >> 16) & below) * tabs_per_row;
            const uint32_t lowb = bd & below;
            const uint32_t start = (uint32_t)((lowb ? p0 + (31 - __clz(lowb)) : pb_j) + 1);
            uint32_t len = (uint32_t)(p0 + i) - start;
            if (col >= A.ncols) {  // (a malformed row is reported through bad_row)
              col = 0;
              len = 0;
            } else if (A.trim) {
              len = trimmed_len(A.buf, start, len);
            }
            W.start[qb + k] = start;
            W.len[qb + k] = len;
            W.col[qb + k] = col;
          }
        }
      }
      __syncwarp();
    }
    // ---- work off full batches (in the extra round: whatever is left, and the side queue)
    const uint32_t have = c.ne - qbase;
    uint32_t off = 0;
    bool flushed = false;
    while (off + 32u <= have || (last && !flushed)) {
      const uint32_t cnt = min(32u, have - off);
      flushed = last && off + cnt == have;
      p1_process<0>(A, wlast, W, off, cnt, qbase + off, nullptr, st, Q, flushed);
      off += cnt;
    }
    if (last) break;
    if (off) {
      __syncwarp();
      const uint32_t left = have - off;  // < 32
      uint32_t a = 0, b = 0, d = 0;
      if (lane < left) {
        a = W.start[off + lane];
        b = W.len[off + lane];
        d = W.col[off + lane];
      }
      __syncwarp();
      if (lane < left) {
        W.start[lane] = a;
        W.len[lane] = b;
        W.col[lane] = d;
      }
      qbase += off;
    }
    __syncwarp();
  }
  // ---- warp totals
  st.max_line = __reduce_max_sync(0xffffffffu, st.max_line);
  st.max_len = __reduce_max_sync(0xffffffffu, st.max_len);
  st.new_count = __reduce_add_sync(0xffffffffu, st.new_count);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) st.new_bytes += __shfl_xor_sync(0xffffffffu, st.new_bytes, o);
  if (lane == 0) {
    if (st.max_line) atomicMax(&A.meta->max_line, st.max_line);
    if (st.new_count) {
      atomicAdd(&A.meta->n_unique, (unsigned long long)st.new_count);
      atomicAdd(&A.meta->dict_str_bytes, st.new_bytes);
      atomicMax(&A.meta->max_str_len, st.max_len);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// pass 1, row-delta variant (wide rows)
//
// The reference parses every field of every row twice (parseInput ConvertToZDW.cpp:329-414, writeBlockRows :486-606).
// What its output depends on is much less: a field whose bytes equal the bytes of the same column in the row before
// has the same value as that row - it is in the dictionary already, inside the column's min/max already, and pass 2 will
// find it equal to the previous value (:532,548,567) and emit nothing.  On analytics-shaped rows (config C3/C4) 84 % of
// the non-empty cells are such repeats.  This variant therefore works on ROWS: a warp owns the rows that start inside
// its tile, reads the row in front of its first one as a reference, and for every row compares each non-empty field with
// the same column of the previous row (column -> field through a non-empty bitmap and its rank prefix).  Only fields that
// CHANGED are parsed / inserted into the hash set, and only they - plus columns that went from a value to empty - leave
// a record (column, value) for pass 2.  A block starts from all-empty columns (:504-505), so the first row is compared
// with an empty row and every distinct field of the block is seen as "changed" at least once.
//
// Byte classification is the same as scan_step's (escape parity, blank lines); positions of the non-empty fields come
// out of it without any search: the k-th field START (a content byte behind a boundary) pairs with the k-th CLOSING
// delimiter behind a content byte, so both are dropped into per-row lists at their ordinals.
// ---------------------------------------------------------------------------------------------
constexpr uint32_t DTILE = 32768;       // bytes of TSV whose row starts one warp owns (small inputs: less, see the driver)
constexpr uint32_t DSTEP = 1024;        // bytes per warp step: 32 lanes x 32 bytes
constexpr uint32_t DCAP = 280;          // non-empty fields of a row a warp can hold (else: delta_bail)
constexpr uint32_t DBW = 128;           // bitmap words per row: up to 4096 columns
constexpr uint32_t DELTA_MAX_COLS = DBW * 32;
constexpr uint32_t DQN = 64;            // changed fields waiting for the full treatment (31 left over + 32 new)
constexpr uint32_t CMP_INLINE = 16;     // fields up to this length are compared straight-line by their lane
constexpr int D1_WARPS = 4;
constexpr int D1_THREADS = D1_WARPS * 32;

struct D1Warp {
  uint16_t S[2][DCAP];   // first byte of the k-th non-empty field, relative to the row start
  uint16_t E[2][DCAP];   // its closing delimiter, relative to the row start
  uint16_t C[DCAP];      // its column (current row only)
  uint16_t PD[DCAP];     // fields whose comparison needs more than CMP_INLINE bytes (worked off together per row)
  uint16_t PF[2][DBW];   // fields in front of bitmap word w
  uint32_t BM[2][DBW];   // bit c = column c of the row is non-empty
  uint32_t CM[(DCAP + 31) / 32];  // bit k & 31 of word k >> 5 = field k changed
};

struct D1Args {
  P1Args P;              // buf, n, lo, limit, ncols, types, trim, hash set, column statistics, rec_col / rec_val, meta
  uint32_t ntiles;       // tiles of tile_bytes bytes
  uint32_t tile_bytes;   // DTILE, or a smaller power of two when the input is too small to fill the GPU with DTILE tiles
  uint32_t nrows;        // rows of the block: the spilled row beyond it has records but no row entry
  uint32_t rec_cap;      // capacity of the record arrays
  uint32_t* row_cnt;     // [nrows] records of row r (low 16 bits; they start at P.row_rec[r]), the first (high 16 bits)
                         // of which are its "became empty" records: two runs, each in column order
  uint32_t* chg_start;   // [rec_cap] where the changed field of record k starts in the TSV ...
  uint32_t* chg_len;     // ... and its length; 0 = the record of a column that became empty (value 0)
  // census-free mode only: row j of tile t goes to slot t * slot_cap + j of P.row_rec / row_cnt
  uint32_t slot_cap;     // row slots per tile
  uint32_t* tile_rows;   // [ntiles] complete rows that start in the tile
};

// Row census of the delta path: per tile the number of row terminators, the last row break and the last row start.
// Only newlines (and a backslash in front of one) matter, so the pass runs at the speed of the read: every warp streams
// its tile through a two-stage ring in shared memory, filled by 1-D bulk copies (TMA, cp.async.bulk + mbarrier) that run
// two chunks ahead of the lanes' 16-byte shared-memory loads.
constexpr uint32_t CEN_CHUNK = 2048;  // bytes per bulk copy (four warp steps)
__global__ void __launch_bounds__(ENC_THREADS)
    k_row_census(const uint8_t* __restrict__ buf, uint64_t n, int64_t lo, uint32_t ntiles, uint32_t tile_bytes, TileAgg* __restrict__ agg) {
  __shared__ __align__(128) uint8_t ring[ENC_WARPS][2][CEN_CHUNK];
  __shared__ __align__(8) uint64_t bars[ENC_WARPS][2];
  const unsigned lane = lane_id(), warp = threadIdx.x >> 5;
  if (lane == 0) {
    mbar_init(&bars[warp][0], 1);
    mbar_init(&bars[warp][1], 1);
  }
  fence_proxy_async();
  __syncthreads();
  const uint32_t tile = blockIdx.x * ENC_WARPS + warp;
  if (tile >= ntiles) return;
  const int64_t t0 = lo + (int64_t)tile * tile_bytes, limit = (int64_t)n;
  // chunks of the tile that hold bytes of the buffer; a chunk's copy ends at the 16-byte boundary behind the last byte
  const int64_t tile_stop = t0 + (int64_t)tile_bytes < limit ? t0 + (int64_t)tile_bytes : limit;
  const uint32_t nchunks = tile_stop > t0 ? (uint32_t)((tile_stop - t0 + CEN_CHUNK - 1) / CEN_CHUNK) : 0u;
  auto issue = [&](uint32_t c) {  // lane 0 only
    const int64_t at = t0 + (int64_t)c * CEN_CHUNK;
    const int64_t left = limit - at;
    const uint32_t bytes = left >= (int64_t)CEN_CHUNK ? CEN_CHUNK : (uint32_t)((left + 15) & ~(int64_t)15);
    mbar_expect_tx(&bars[warp][c & 1u], bytes);
    bulk_load(ring[warp][c & 1u], buf + at, bytes, &bars[warp][c & 1u]);
  };
  if (lane == 0) {
    if (nchunks > 0) issue(0);
    if (nchunks > 1) issue(1);
  }
  uint32_t c_nl = t0 <= 0 ? 1u : (is_unescaped_newline(buf, t0 - 1) ? 1u : 0u);
  uint32_t rows = 0;
  int32_t last_r = -1, last_s = -1;
  for (uint32_t c = 0; c < nchunks; ++c) {
    mbar_wait(&bars[warp][c & 1u], (c >> 1) & 1u);
    const uint8_t* stage = ring[warp][c & 1u];
    for (uint32_t q = 0; q < CEN_CHUNK; q += STEP) {
      const uint32_t s = c * CEN_CHUNK + q;
      const int64_t p0 = t0 + s + 16 * (int64_t)lane;
      uint32_t nl = 0, in = 0;
      if (p0 < limit && p0 + 16 > 0) {
        const uint4 v = *reinterpret_cast<const uint4*>(stage + q + 16u * lane);
        const int64_t ia = p0 < 0 ? -p0 : 0;
        const int64_t ib = p0 + 16 > limit ? limit - p0 : 16;
        in = ((1u << ib) - 1u) & ~((1u << ia) - 1u);
        if (chunk_has(v, '\n')) {
          nl = chunk_mask(v, '\n') & in;
          uint32_t m = nl;
          while (m) {  // escape parity (getnextrow.cpp:44-53): rare, walked byte by byte
            const int i = __ffs(m) - 1;
            m &= m - 1;
            if (odd_backslashes_before(buf, p0 + i)) nl &= ~(1u << i);
          }
        }
      }
      uint32_t prevnl = __shfl_up_sync(0xffffffffu, nl >> 15, 1);
      if (lane == 0) prevnl = c_nl;
      uint32_t after_nl = ((nl << 1) | prevnl) & 0xffffu;
      if (p0 <= 0 && p0 + 16 > 0) after_nl |= 1u << (-p0);
      const uint32_t skip = nl & after_nl, term = nl & ~skip, rs = after_nl & ~nl & in;
      rows += (uint32_t)__popc(term);
      if (nl) last_r = (int32_t)(s + 16u * lane) + (31 - __clz(nl));
      if (rs) last_s = (int32_t)(s + 16u * lane) + (31 - __clz(rs));
      c_nl = __shfl_sync(0xffffffffu, nl >> 15, 31);
    }
    __syncwarp();  // every lane has its bytes of the stage in registers: it can be filled again
    if (lane == 0 && c + 2 < nchunks) {
      fence_proxy_async();
      issue(c + 2);
    }
  }
  rows = __reduce_add_sync(0xffffffffu, rows);
  last_r = __reduce_max_sync(0xffffffffu, last_r);
  last_s = __reduce_max_sync(0xffffffffu, last_s);
  if (lane == 0) {
    TileAgg a;
    a.rows = rows;
    a.tabs = 0;
    a.ne = 0;
    a.break_p1 = last_r >= 0 ? (uint32_t)(t0 + last_r + 1) : 0u;
    a.bound_p1 = a.break_p1;
    a.rs_p1 = last_s >= 0 ? (uint32_t)(t0 + last_s + 1) : 0u;
    agg[tile] = a;
  }
}

// 32-bit masks of a lane's 32 bytes: bit i = byte i equals `ch`.  bytes_eq leaves 0x80 in every matching byte; a dot
// product with the byte weights 1, 2, 4, ... gathers the four flags of a word, two words per accumulator.
__device__ __forceinline__ uint32_t mask16_dp(const uint4& v, uint32_t rep) {
  const uint32_t lo = __dp4a(bytes_eq(v.x, rep), 0x08040201u, __dp4a(bytes_eq(v.y, rep), 0x80402010u, 0u));
  const uint32_t hi = __dp4a(bytes_eq(v.z, rep), 0x08040201u, __dp4a(bytes_eq(v.w, rep), 0x80402010u, 0u));
  return (lo >> 7) | (hi << 1);  // both sums carry the factor 0x80
}
__device__ __forceinline__ uint32_t mask32(const uint4& a, const uint4& b, uint8_t ch) {
  const uint32_t rep = 0x01010101u * ch;
  return mask16_dp(a, rep) | (mask16_dp(b, rep) << 16);
}

// lane's 32-bit mask of the step's bit positions >= a / <= b (positions 0..1023, lane l holds 32 l .. 32 l + 31)
__device__ __forceinline__ uint32_t lane_bits_ge(int32_t a, unsigned lane) {
  const int32_t lo = a - (int32_t)(lane * 32u);
  return lo <= 0 ? 0xffffffffu : (lo >= 32 ? 0u : (0xffffffffu << lo));
}
__device__ __forceinline__ uint32_t lane_bits_le(int32_t b, unsigned lane) {
  const int32_t hi = b - (int32_t)(lane * 32u);
  return hi < 0 ? 0u : (hi >= 31 ? 0xffffffffu : ((2u << hi) - 1u));
}
__device__ __forceinline__ uint32_t bits_below(uint32_t i) { return (1u << i) - 1u; }  // i < 32

// do the `len` (1..16) bytes at a and b differ?  Straight-line: five aligned words a side, funnel shifts, one mask.
// SAFE = both fields lie at least 20 bytes in front of the end of the buffer: no load needs clamping.
template <bool SAFE>
__device__ __forceinline__ bool short_differ(const uint8_t* __restrict__ a, const uint8_t* __restrict__ b, uint32_t len,
                                             const uint32_t* wlast) {
  const uintptr_t ua = reinterpret_cast<uintptr_t>(a), ub = reinterpret_cast<uintptr_t>(b);
  const uint32_t* wa = reinterpret_cast<const uint32_t*>(ua & ~(uintptr_t)3);
  const uint32_t* wb = reinterpret_cast<const uint32_t*>(ub & ~(uintptr_t)3);
  const uint32_t sa = (uint32_t)(ua & 3u) * 8u, sb = (uint32_t)(ub & 3u) * 8u;
  uint32_t a0, a1, a2, a3, a4, b0, b1, b2, b3, b4;
  if (SAFE) {
    a0 = __ldg(wa), a1 = __ldg(wa + 1), a2 = __ldg(wa + 2), a3 = __ldg(wa + 3), a4 = __ldg(wa + 4);
    b0 = __ldg(wb), b1 = __ldg(wb + 1), b2 = __ldg(wb + 2), b3 = __ldg(wb + 3), b4 = __ldg(wb + 4);
  } else {
    const uint32_t ra = (uint32_t)min((ptrdiff_t)4, wlast - wa), rb = (uint32_t)min((ptrdiff_t)4, wlast - wb);
    a0 = __ldg(wa), a1 = __ldg(wa + min(1u, ra)), a2 = __ldg(wa + min(2u, ra)), a3 = __ldg(wa + min(3u, ra)), a4 = __ldg(wa + min(4u, ra));
    b0 = __ldg(wb), b1 = __ldg(wb + min(1u, rb)), b2 = __ldg(wb + min(2u, rb)), b3 = __ldg(wb + min(3u, rb)), b4 = __ldg(wb + min(4u, rb));
  }
  const uint32_t x0 = __funnelshift_r(a0, a1, sa) ^ __funnelshift_r(b0, b1, sb);
  const uint32_t x1 = __funnelshift_r(a1, a2, sa) ^ __funnelshift_r(b1, b2, sb);
  const uint32_t x2 = __funnelshift_r(a2, a3, sa) ^ __funnelshift_r(b2, b3, sb);
  const uint32_t x3 = __funnelshift_r(a3, a4, sa) ^ __funnelshift_r(b3, b4, sb);
  // keep the first len bytes: word w keeps min(4, len - 4 w) of them
  const uint32_t tail = len & 3u, tm = tail ? ((1u << (8u * tail)) - 1u) : 0xffffffffu, nw = (len + 3u) >> 2;
  uint32_t d = x0 & (nw == 1u ? tm : 0xffffffffu);
  if (nw > 1u) d |= x1 & (nw == 2u ? tm : 0xffffffffu);
  if (nw > 2u) d |= x2 & (nw == 3u ? tm : 0xffffffffu);
  if (nw > 3u) d |= x3 & tm;
  return d != 0u;
}

// the same for any length, one lane, 16 bytes a round (used for 17 .. MID_MAX bytes, a row's worth of them side by
// side).  SAFE = both fields end at least 20 bytes in front of the end of the buffer.
template <bool SAFE>
__device__ __forceinline__ bool bytes_differ(const uint8_t* __restrict__ a, const uint8_t* __restrict__ b, uint32_t len,
                                             const uint32_t* wlast) {
  const uintptr_t ua = reinterpret_cast<uintptr_t>(a), ub = reinterpret_cast<uintptr_t>(b);
  const uint32_t* wa = reinterpret_cast<const uint32_t*>(ua & ~(uintptr_t)3);
  const uint32_t* wb = reinterpret_cast<const uint32_t*>(ub & ~(uintptr_t)3);
  const uint32_t sa = (uint32_t)(ua & 3u) * 8u, sb = (uint32_t)(ub & 3u) * 8u;
  uint32_t pa = __ldg(wa), pb = __ldg(wb);
  const uint32_t nw = (len + 3u) >> 2;
  const uint32_t tail = len & 3u, tm = tail ? ((1u << (8u * tail)) - 1u) : 0xffffffffu;
  if (SAFE) {
    for (uint32_t k = 0; k < nw; k += 4u) {
      const uint32_t a1 = __ldg(wa + k + 1), a2 = __ldg(wa + k + 2), a3 = __ldg(wa + k + 3), a4 = __ldg(wa + k + 4);
      const uint32_t b1 = __ldg(wb + k + 1), b2 = __ldg(wb + k + 2), b3 = __ldg(wb + k + 3), b4 = __ldg(wb + k + 4);
      const uint32_t x0 = __funnelshift_r(pa, a1, sa) ^ __funnelshift_r(pb, b1, sb);
      const uint32_t x1 = __funnelshift_r(a1, a2, sa) ^ __funnelshift_r(b1, b2, sb);
      const uint32_t x2 = __funnelshift_r(a2, a3, sa) ^ __funnelshift_r(b2, b3, sb);
      const uint32_t x3 = __funnelshift_r(a3, a4, sa) ^ __funnelshift_r(b3, b4, sb);
      pa = a4;
      pb = b4;
      const uint32_t left = nw - k;  // words of the field in this round (>= 1)
      uint32_t d = x0 & (left == 1u ? tm : 0xffffffffu);
      if (left > 1u) d |= x1 & (left == 2u ? tm : 0xffffffffu);
      if (left > 2u) d |= x2 & (left == 3u ? tm : 0xffffffffu);
      if (left > 3u) d |= x3 & (left == 4u ? tm : 0xffffffffu);
      if (d) return true;
    }
    return false;
  }
  uint32_t diff = 0;
  for (uint32_t k = 0; k < nw && diff == 0u; ++k) {
    const uint32_t* qa = wa + k + 1;
    const uint32_t* qb = wb + k + 1;
    const uint32_t na = __ldg(qa <= wlast ? qa : wlast), nb = __ldg(qb <= wlast ? qb : wlast);
    uint32_t x = __funnelshift_r(pa, na, sa) ^ __funnelshift_r(pb, nb, sb);
    pa = na;
    pb = nb;
    if (k + 1u == nw) x &= tm;
    diff = x;
  }
  return diff != 0u;
}

// ... and by the whole warp, 128 bytes a round, for the rare long field (all lanes call, all get the verdict)
__device__ __forceinline__ bool warp_differ(const uint8_t* __restrict__ a, const uint8_t* __restrict__ b, uint32_t len,
                                            const uint32_t* wlast) {
  const uintptr_t ua = reinterpret_cast<uintptr_t>(a), ub = reinterpret_cast<uintptr_t>(b);
  const uint32_t* wa = reinterpret_cast<const uint32_t*>(ua & ~(uintptr_t)3);
  const uint32_t* wb = reinterpret_cast<const uint32_t*>(ub & ~(uintptr_t)3);
  const uint32_t sa = (uint32_t)(ua & 3u) * 8u, sb = (uint32_t)(ub & 3u) * 8u;
  const uint32_t nw = (len + 3u) >> 2;
  for (uint32_t k0 = 0; k0 < nw; k0 += 32u) {
    const uint32_t k = k0 + lane_id();
    uint32_t x = 0;
    if (k < nw) {
      const uint32_t* qa = wa + k;
      const uint32_t* qb = wb + k;
      x = __funnelshift_r(__ldg(qa), __ldg(qa + 1 <= wlast ? qa + 1 : wlast), sa) ^
          __funnelshift_r(__ldg(qb), __ldg(qb + 1 <= wlast ? qb + 1 : wlast), sb);
      const uint32_t rem = len - 4u * k;
      if (rem < 4u) x &= (1u << (8u * rem)) - 1u;
    }
    if (__any_sync(0xffffffffu, x != 0u)) return true;
  }
  return false;
}

// Where column `col` of the row before (lists of `prv`) lies in the TSV: (start << 32) | len, 0 = it was empty.  Every
// record carries this in its rec_val until k_pass1d_values has compared the two values and put the new one there.
__device__ __forceinline__ unsigned long long d1_prev_field(const D1Warp& W, uint32_t prv, uint32_t col, int64_t prev_start) {
  const uint32_t pw = W.BM[prv][col >> 5], bit = col & 31u;
  if (!((pw >> bit) & 1u)) return 0ull;
  const uint32_t j = (uint32_t)W.PF[prv][col >> 5] + (uint32_t)__popc(pw & bits_below(bit));
  const uint32_t ps = W.S[prv][j];
  return ((unsigned long long)(uint32_t)(prev_start + ps) << 32) | ((uint32_t)W.E[prv][j] - ps);
}

// The open row is complete (n fields in the lists of `cur`, their columns' bits in BM[cur], set while they were
// extracted): rank prefix of the bitmap; unless it is the reference row,
// compare with the row before (lists of cur ^ 1), hand out the records and queue the changed fields.
// r = row number, or >= A.nrows for the spilled row (no row entry: its records only feed the dictionary and the column
// ranges).  The changed fields are only LISTED here (record slot, column, position, length); k_pass1d_values works the
// list off afterwards - two small kernels instead of one that does not fit the instruction cache.
__device__ __forceinline__ void d1_finish_row(const D1Args& A, const uint32_t* wlast, D1Warp& W, uint32_t cur, uint32_t n,
                                              int64_t row_start, int64_t prev_start, bool reference, uint32_t r) {
  const P1Args& P = A.P;
  const unsigned lane = lane_id();
  const uint32_t BW = (P.ncols + 31u) >> 5, prv = cur ^ 1u;
  // ---- -t: trailing spaces do not belong to a field; a field of spaces only is an empty one (ConvertToZDW.cpp:295-313)
  if (P.trim) {  // (the bitmap is rebuilt from the fields that stay)
    for (uint32_t w = lane; w < BW; w += 32u) W.BM[cur][w] = 0u;
    __syncwarp();
    uint32_t kept = 0;
    for (uint32_t k0 = 0; k0 < n; k0 += 32u) {
      const uint32_t k = k0 + lane;
      uint32_t s = 0, e = 0, c = 0;
      if (k < n) {
        s = W.S[cur][k];
        e = W.E[cur][k];
        c = W.C[k];
        while (e > s && __ldg(P.buf + row_start + e - 1) == (uint8_t)' ') --e;
      }
      const unsigned m = __ballot_sync(0xffffffffu, e > s);
      __syncwarp();
      if (e > s) {
        const uint32_t d = kept + (uint32_t)__popc(m & lanemask_lt());
        W.S[cur][d] = (uint16_t)s;
        W.E[cur][d] = (uint16_t)e;
        W.C[d] = (uint16_t)c;
        atomicOr(&W.BM[cur][c >> 5], 1u << (c & 31u));
      }
      kept += (uint32_t)__popc(m);
      __syncwarp();
    }
    n = kept;
  }
  // ---- rank prefix: fields in front of every bitmap word
  {
    uint32_t run = 0;
    for (uint32_t w0 = 0; w0 < BW; w0 += 32u) {
      const uint32_t w = w0 + lane;
      const uint32_t c = w < BW ? (uint32_t)__popc(W.BM[cur][w]) : 0u;
      uint32_t inc = c;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= (unsigned)o) inc += t;
      }
      if (w < BW) W.PF[cur][w] = (uint16_t)(run + inc - c);
      run += __shfl_sync(0xffffffffu, inc, 31);
    }
  }
  __syncwarp();
  if (reference) return;

  // ---- which fields changed?  Up to CMP_INLINE bytes are compared on the spot; longer fields of equal length are
  // listed and compared together afterwards (one lane each, so that no lane drags a 100-byte loop through a batch of
  // 8-byte fields).  CM[b] = verdicts of batch b.
  uint32_t nchg = 0, npd = 0;
  // both rows end far enough from the end of the buffer (a row is at most 64 KiB long): the compares need no clamping
  const bool safe = (uint64_t)row_start + 65536u + 32u < P.n && (uint64_t)prev_start + 65536u + 32u < P.n;
  for (uint32_t k0 = 0, b = 0; k0 < n; k0 += 32u, ++b) {
    const uint32_t k = k0 + lane;
    bool changed = false, pending = false;
    if (k < n) {
      const uint32_t s = W.S[cur][k], len = (uint32_t)W.E[cur][k] - s, col = W.C[k];
      const uint32_t pw = W.BM[prv][col >> 5], bit = col & 31u;
      changed = true;
      if ((pw >> bit) & 1u) {
        const uint32_t j = (uint32_t)W.PF[prv][col >> 5] + (uint32_t)__popc(pw & bits_below(bit));
        const uint32_t ps = W.S[prv][j], pl = (uint32_t)W.E[prv][j] - ps;
        if (pl == len) {
          if (len <= CMP_INLINE) {
            changed = safe ? short_differ<true>(P.buf + row_start + s, P.buf + prev_start + ps, len, wlast)
                           : short_differ<false>(P.buf + row_start + s, P.buf + prev_start + ps, len, wlast);
          } else {
            changed = false;
            pending = true;
          }
        }
      }
    }
    const unsigned m = __ballot_sync(0xffffffffu, changed), mp = __ballot_sync(0xffffffffu, pending);
    if (lane == 0) W.CM[b] = m;
    if (pending) W.PD[npd + (uint32_t)__popc(mp & lanemask_lt())] = (uint16_t)k;
    nchg += (uint32_t)__popc(m);
    npd += (uint32_t)__popc(mp);
  }
  __syncwarp();
  for (uint32_t q0 = 0; q0 < npd; q0 += 32u) {
    const uint32_t q = q0 + lane;
    bool changed = false, big = false;
    uint32_t k = 0, s = 0, len = 0, ps = 0;
    if (q < npd) {
      k = W.PD[q];
      s = W.S[cur][k];
      len = (uint32_t)W.E[cur][k] - s;
      const uint32_t col = W.C[k];
      const uint32_t pw = W.BM[prv][col >> 5], bit = col & 31u;
      ps = W.S[prv][(uint32_t)W.PF[prv][col >> 5] + (uint32_t)__popc(pw & bits_below(bit))];
      if (len <= MID_MAX) {
        changed = safe ? bytes_differ<true>(P.buf + row_start + s, P.buf + prev_start + ps, len, wlast)
                       : bytes_differ<false>(P.buf + row_start + s, P.buf + prev_start + ps, len, wlast);
      } else {
        big = true;
      }
    }
    unsigned todo = __ballot_sync(0xffffffffu, big);
    while (todo) {  // the rare long field: the whole warp compares it
      const int src = __ffs(todo) - 1;
      todo &= todo - 1;
      const uint32_t s2 = __shfl_sync(0xffffffffu, s, src), p2 = __shfl_sync(0xffffffffu, ps, src),
                     l2 = __shfl_sync(0xffffffffu, len, src);
      const bool d = warp_differ(P.buf + row_start + s2, P.buf + prev_start + p2, l2, wlast);
      if ((int)lane == src) changed = d;
    }
    if (changed) atomicOr(&W.CM[k >> 5], 1u << (k & 31u));
    nchg += (uint32_t)__popc(__ballot_sync(0xffffffffu, changed));
  }
  __syncwarp();
  // ---- columns that had a value in the row before and are empty now
  uint32_t nte = 0;
  for (uint32_t w = lane; w < BW; w += 32u) nte += (uint32_t)__popc(W.BM[prv][w] & ~W.BM[cur][w]);
  nte = __reduce_add_sync(0xffffffffu, nte);
  const uint32_t cnt = nchg + nte;
  // ---- records of the row: one bump allocation
  uint32_t base = 0;
  if (lane == 0 && cnt) base = atomicAdd(&P.meta->rec_count, cnt);
  base = __shfl_sync(0xffffffffu, base, 0);
  bool drop = false;
  if (cnt && (base > A.rec_cap || cnt > A.rec_cap - base)) {
    if (lane == 0) *reinterpret_cast<volatile uint32_t*>(&P.meta->rec_overflow) = 1u;
    drop = true;
  }
  if (r < A.nrows && lane == 0) {
    P.row_rec[r] = base;
    A.row_cnt[r] = drop ? 0u : cnt | (nte << 16);
  }
  if (drop || !cnt) return;
  // ---- "became empty" records: (column, the field it had in the row before)
  if (nte) {
    uint32_t run = 0;
    for (uint32_t w0 = 0; w0 < BW; w0 += 32u) {
      const uint32_t w = w0 + lane;
      uint32_t x = w < BW ? (W.BM[prv][w] & ~W.BM[cur][w]) : 0u;
      const uint32_t c = (uint32_t)__popc(x);
      uint32_t inc = c;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= (unsigned)o) inc += t;
      }
      uint32_t at = base + run + inc - c;
      while (x) {
        const uint32_t bit = (uint32_t)__ffs(x) - 1u;
        x &= x - 1u;
        P.rec_col[at] = w * 32u + bit;
        P.rec_val[at] = d1_prev_field(W, prv, w * 32u + bit, prev_start);
        A.chg_len[at] = 0u;
        ++at;
      }
      run += __shfl_sync(0xffffffffu, inc, 31);
    }
  }
  // ---- changed fields: listed with the record each of them fills
  uint32_t at = base + nte;
  for (uint32_t k0 = 0, b = 0; k0 < n && nchg; k0 += 32u, ++b) {
    const unsigned m = W.CM[b];
    if (!m) continue;
    const uint32_t k = k0 + lane;
    if ((m >> lane) & 1u) {
      const uint32_t s = W.S[cur][k], d = at + (uint32_t)__popc(m & lanemask_lt()), col = W.C[k];
      P.rec_col[d] = col;
      P.rec_val[d] = d1_prev_field(W, prv, col, prev_start);
      A.chg_start[d] = (uint32_t)(row_start + s);
      A.chg_len[d] = (uint32_t)W.E[cur][k] - s;
    }
    at += (uint32_t)__popc(m);
  }
}

// Census-free mode: position + 1 of the last row start in front of t0 (a byte other than '\n' behind an unescaped
// newline, or the buffer's first byte), which is what the census's prefix of rs_p1 holds for the tile; 0 = only blank
// lines in front of t0.  The warp walks back from t0 a step at a time and looks at newlines only.  -1: no row starts
// within 64 KiB plus a step, the delta path's row limit (the warp bails; the host runs the block with the census).
__device__ __forceinline__ int64_t d1_ref_start_p1(const uint8_t* __restrict__ buf, int64_t t0, unsigned lane) {
  uint32_t nl_behind = 1u;  // the byte behind the step is '\n' - or is t0, where a row start does not count
  for (int64_t hi = t0; hi > 0; hi -= DSTEP) {
    if (t0 - hi > 65536) return -1;
    const int64_t p0 = hi - (int64_t)DSTEP + 32 * (int64_t)lane;  // (16-byte aligned in memory, as the tiles are)
    uint32_t nl = 0;
    if (p0 + 32 > 0) {
      const uint4 v0 = p0 + 16 > 0 ? ldg_keep_u4(buf + p0) : make_uint4(0u, 0u, 0u, 0u);
      const uint4 v1 = ldg_keep_u4(buf + p0 + 16);
      if (chunk_has(v0, '\n') || chunk_has(v1, '\n'))
        nl = mask32(v0, v1, '\n') & (p0 >= 0 ? 0xffffffffu : ~bits_below((uint32_t)-p0));
    }
    uint32_t behind = __shfl_down_sync(0xffffffffu, nl & 1u, 1);
    if (lane == 31) behind = nl_behind;
    nl_behind = __shfl_sync(0xffffffffu, nl & 1u, 0);
    uint32_t brk = nl & ~((nl >> 1) | (behind << 31));  // newlines followed by a byte other than '\n'
    for (uint32_t m = brk; m; m &= m - 1u) {  // escape parity: rare, walked byte by byte
      const int i = __ffs(m) - 1;
      if (odd_backslashes_before(buf, p0 + i)) brk &= ~(1u << i);
    }
    const int32_t best = __reduce_max_sync(0xffffffffu, brk ? (int32_t)(lane * 32u) + (31 - __clz(brk)) : -1);
    if (best >= 0) return hi - (int64_t)DSTEP + best + 2;
    if (hi <= (int64_t)DSTEP) return __ldg(buf) != (uint8_t)'\n' ? 1 : 0;  // the step holds the buffer's first byte
  }
  return 0;
}

// CF = census-free: no TileAgg prefix.  The warp finds its reference row itself (d1_ref_start_p1), numbers the rows it
// owns from 0 into its tile's slots, and reports the last row break it saw; k_row_fixup makes the numbers global.  The
// limit is the end of the buffer, and a row it cuts short is dropped (it is the unterminated tail).
template <bool CF>
__global__ void __launch_bounds__(D1_THREADS, 8) k_pass1d(const D1Args A) {
  __shared__ D1Warp sw[D1_WARPS];
  const P1Args& P = A.P;
  const unsigned lane = lane_id(), warp = threadIdx.x >> 5;
  const uint32_t tile = blockIdx.x * D1_WARPS + warp;
  if (tile >= A.ntiles) return;
  const int64_t t0 = P.lo + (int64_t)tile * A.tile_bytes;
  if (t0 >= P.limit) {
    if (CF && lane == 0) A.tile_rows[tile] = 0u;
    return;
  }
  const int64_t tile_end = t0 + A.tile_bytes;
  D1Warp& W = sw[warp];
  const uint32_t* wlast = reinterpret_cast<const uint32_t*>(reinterpret_cast<uintptr_t>(P.buf + P.n - 1) & ~(uintptr_t)3);
  TileAgg pre;
  if (CF) {
    const int64_t rs_p1 = d1_ref_start_p1(P.buf, t0, lane);
    if (rs_p1 < 0) {
      if (lane == 0) *reinterpret_cast<volatile uint32_t*>(&P.meta->delta_bail) = 1u;
      return;
    }
    pre.rs_p1 = (uint32_t)rs_p1;
    pre.rows = 0u;
  } else {
    pre = P.pre[tile];
  }
  const uint32_t BW = (P.ncols + 31u) >> 5;
  // the row in front of the tile's first row (if there is one) is read as the reference the first row is compared with
  const bool have_prev = pre.rs_p1 != 0u;
  const int64_t scan_from = have_prev ? (int64_t)pre.rs_p1 - 1 : (t0 > 0 ? t0 : 0);
  uint32_t last_nl_p1 = 0;  // CF: position + 1 of the last row break the lane saw
  for (uint32_t w = lane; w < BW; w += 32u) W.BM[0][w] = W.BM[1][w] = 0u;  // "the row before" of a block's first row is empty
  __syncwarp();
  const uint32_t tabs_per_row = P.ncols - 1u;
  uint32_t max_line = 0;

  uint32_t cur = 0;
  bool row_open = false, reference = false;
  int64_t row_start = 0, prev_start = 0;
  uint32_t n_ne = 0, tabs = 0, row_no = 0, rows_seen = 0;
  uint32_t c_bs = 0, c_nl = 0, c_bd = 0;
  bool bail = false;

  int64_t sb = scan_from - ((scan_from - P.lo) & 15);  // step positions are 16-byte aligned in memory
  int64_t c_lastb = scan_from - 1;                     // the last boundary in front of the step (the scan starts behind a row break)
  // One loop, one call site for the row work (the kernel must stay small: it is instruction-cache sensitive).  Every
  // round either completes a row (need_finish), fetches the next 1 KiB step, or handles the step's next event.
  bool have_step = false, need_finish = false, final = false, stop = false, first = true, plain = false;
  uint32_t fin_row = 0;
  uint32_t tab = 0, term = 0, bound = 0, ne = 0, rs = 0;
  int32_t lb_in = 0, cursor = 0;
  for (;;) {
    if (need_finish) {
      d1_finish_row(A, wlast, W, cur, n_ne, row_start, prev_start, reference, fin_row);
      need_finish = false;
      if (final) break;
      prev_start = row_start;
      cur ^= 1u;
      row_open = false;
    }
    if (!have_step) {
      if (bail) break;
      if (stop || sb >= P.limit || (!row_open && sb >= tile_end)) {
        // a row the block's limit cut short (the reference's interrupted row, SURVEY App. B-14): the columns in front
        // of the limit count for the dictionary and the column ranges, the row itself is not part of the block
        if (!CF && row_open && !reference && n_ne) {
          need_finish = final = true;
          fin_row = 0xffffffffu;
          continue;
        }
        break;
      }
      const int64_t p0 = sb + 32 * (int64_t)lane;
      uint32_t nl = 0, bs = 0, in = 0;
      tab = 0;
      if (p0 < P.limit && p0 + 32 > scan_from) {
        const uint4 v0 = ldg_keep_u4(P.buf + p0);
        const uint4 v1 = p0 + 16 < P.limit ? ldg_keep_u4(P.buf + p0 + 16) : make_uint4(0u, 0u, 0u, 0u);
        if (p0 + 2 * (int64_t)DSTEP < P.limit) prefetch_l2(P.buf + p0 + 2 * DSTEP);  // (measured: 0.983 -> 0.961 ms per C4 block)
        in = 0xffffffffu;
        if (sb < scan_from || sb + (int64_t)DSTEP > P.limit) {  // (warp-uniform: only the first and the last step)
          const int64_t ia = p0 < scan_from ? scan_from - p0 : 0;
          const int64_t ib = p0 + 32 > P.limit ? P.limit - p0 : 32;
          in = (ib >= 32 ? 0xffffffffu : ((1u << ib) - 1u)) & ~((1u << ia) - 1u);
        }
        tab = mask32(v0, v1, '\t') & in;
        if (chunk_has(v0, '\n') || chunk_has(v1, '\n')) nl = mask32(v0, v1, '\n') & in;
        if (chunk_has(v0, '\\') || chunk_has(v1, '\\')) bs = mask32(v0, v1, '\\') & in;
      }
      {  // escape parity: only delimiters that directly follow a backslash need the backward walk
        uint32_t prev = __shfl_up_sync(0xffffffffu, bs >> 31, 1);
        if (lane == 0) prev = c_bs;
        uint32_t sus = (tab | nl) & ((bs << 1) | prev);
        while (sus) {
          const int i = __ffs(sus) - 1;
          sus &= sus - 1;
          if (odd_backslashes_before(P.buf, p0 + i)) {
            tab &= ~(1u << i);
            nl &= ~(1u << i);
          }
        }
      }
      if (CF && nl) last_nl_p1 = (uint32_t)(p0 + 32 - __clz(nl));
      const uint32_t fix = (first && p0 <= scan_from && p0 + 32 > scan_from) ? 1u << (scan_from - p0) : 0u;
      uint32_t prevnl = __shfl_up_sync(0xffffffffu, nl >> 31, 1);
      if (lane == 0) prevnl = c_nl;
      const uint32_t after_nl = ((nl << 1) | prevnl) | fix;
      const uint32_t skip = nl & after_nl;
      term = nl & ~skip;
      bound = tab | nl;
      uint32_t prevbd = __shfl_up_sync(0xffffffffu, bound >> 31, 1);
      if (lane == 0) prevbd = c_bd;
      const uint32_t after_bound = ((bound << 1) | prevbd) | fix;
      ne = (tab | term) & ~after_bound;   // closing delimiters of non-empty fields
      rs = after_nl & ~nl & in;           // first bytes of rows
      c_bs = __shfl_sync(0xffffffffu, bs >> 31, 31);
      c_nl = __shfl_sync(0xffffffffu, nl >> 31, 31);
      c_bd = __shfl_sync(0xffffffffu, bound >> 31, 31);
      {  // the last boundary in front of every lane's bytes, as a step position (negative: in an earlier step)
        const int32_t mine = bound ? (int32_t)(lane * 32u) + (31 - __clz(bound)) : INT32_MIN;
        int32_t inc = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int32_t t = __shfl_up_sync(0xffffffffu, inc, o);
          if (lane >= (unsigned)o) inc = max(inc, t);
        }
        lb_in = __shfl_up_sync(0xffffffffu, inc, 1);
        if (lane == 0) lb_in = INT32_MIN;
        lb_in = max(lb_in, (int32_t)(c_lastb - sb));
        const int32_t top = __shfl_sync(0xffffffffu, inc, 31);
        if (top != INT32_MIN) c_lastb = sb + top;
      }
      plain = row_open && __ballot_sync(0xffffffffu, nl != 0u) == 0u;  // the usual step of a wide row
      cursor = 0;
      have_step = true;
      first = false;
    }
    // ---- the step's next event: a row start opens a row, a terminator completes it
    if (!row_open) {
      const uint32_t m = rs & lane_bits_ge(cursor, lane);
      const unsigned b = __ballot_sync(0xffffffffu, m != 0u);
      if (!b) {
        have_step = false;
        sb += DSTEP;
        continue;
      }
      const int src = __ffs(b) - 1;
      const int32_t pos = src * 32 + (__ffs(__shfl_sync(0xffffffffu, m, src)) - 1);
      const int64_t start_abs = sb + pos;
      if (start_abs >= tile_end) {  // the next warp's row: done
        stop = true;
        have_step = false;
        continue;
      }
      row_open = true;
      reference = start_abs < t0;
      row_start = start_abs;
      row_no = CF ? rows_seen : pre.rows + rows_seen;
      n_ne = tabs = 0;
      cursor = pos;
      for (uint32_t w = lane; w < BW; w += 32u) W.BM[cur][w] = 0u;  // (filled while the fields are extracted)
      __syncwarp();
    }
    int32_t seg_end = (int32_t)DSTEP - 1;
    bool ends = false;
    if (!plain) {
      const uint32_t m = term & lane_bits_ge(cursor, lane);
      const unsigned b = __ballot_sync(0xffffffffu, m != 0u);
      if (b) {
        const int src = __ffs(b) - 1;
        seg_end = src * 32 + (__ffs(__shfl_sync(0xffffffffu, m, src)) - 1);
        ends = true;
      }
    }
    // ---- the fields that close in [cursor, seg_end]: every lane drops the positions of its closing delimiters into
    // the row's list at their ordinals; then field k is worked out by lane k & 31 - column from the tabs in front of
    // it, first byte from the last boundary in front of it
    {
      const uint32_t seg = plain ? 0xffffffffu : (lane_bits_ge(cursor, lane) & lane_bits_le(seg_end, lane));
      uint32_t e_ = ne & seg;
      const uint32_t t_ = tab & seg;
      const uint32_t mine = (uint32_t)__popc(e_) | ((uint32_t)__popc(t_) << 16);
      uint32_t inc = mine;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= (unsigned)o) inc += t;
      }
      const uint32_t ex = inc - mine, tot = __shfl_sync(0xffffffffu, inc, 31);
      const uint32_t nf = tot & 0xffffu;
      // does everything fit?  (field positions are 16-bit, relative to the row start)
      if (n_ne + nf > DCAP || sb + (int64_t)DSTEP - row_start > 65535) {
        bail = true;
        have_step = false;
        continue;
      }
      const int32_t rel_sb = (int32_t)(sb - row_start);  // step position -> row-relative position
      uint32_t oe = n_ne + (ex & 0xffffu);
      while (e_) {
        const uint32_t i = (uint32_t)__ffs(e_) - 1u;
        e_ &= e_ - 1u;
        W.E[cur][oe++] = (uint16_t)(rel_sb + (int32_t)(lane * 32u + i));
      }
      __syncwarp();
      const uint32_t tb = tabs + (ex >> 16);
      for (uint32_t k0 = 0; k0 < nf; k0 += 32u) {
        const uint32_t k = n_ne + k0 + lane;
        const bool mine_f = k0 + lane < nf;
        const int32_t pos = mine_f ? (int32_t)W.E[cur][k] - rel_sb : 0;
        const int j = pos >> 5;
        const uint32_t i = (uint32_t)pos & 31u;
        const uint32_t tj = __shfl_sync(0xffffffffu, t_, j), bj = __shfl_sync(0xffffffffu, bound, j);
        const uint32_t tbj = __shfl_sync(0xffffffffu, tb, j);
        const int32_t lbj = __shfl_sync(0xffffffffu, lb_in, j);
        if (mine_f) {
          const uint32_t lowb = bj & bits_below(i);
          const int32_t fs = (lowb ? j * 32 + (31 - __clz(lowb)) : lbj) + 1;
          W.S[cur][k] = (uint16_t)(rel_sb + fs);
          const uint32_t col = min(tbj + (uint32_t)__popc(tj & bits_below(i)), P.ncols - 1u);
          W.C[k] = (uint16_t)col;
          atomicOr(&W.BM[cur][col >> 5], 1u << (col & 31u));
        }
      }
      n_ne += nf;
      tabs += tot >> 16;
    }
    __syncwarp();
    if (!ends) {
      have_step = false;
      sb += DSTEP;
      continue;
    }
    // ---- the row is complete
    const int64_t term_abs = sb + seg_end;
    if (!reference) {
      if (tabs != tabs_per_row) {  // ConvertToZDW.cpp:336-337
        if (CF) {
          if (lane == 0) atomicMin(&P.meta->bad_slot, ((unsigned long long)tile << 32) | row_no);
        } else {
          atomicMin(&P.meta->bad_row, row_no);
        }
      }
      max_line = max(max_line, (uint32_t)(term_abs - row_start + 1));
    }
    fin_row = row_no;
    if (CF) {  // rows_seen counts the rows the tile owns
      if (!reference) {
        ++rows_seen;
        fin_row = row_no < A.slot_cap ? tile * A.slot_cap + row_no : 0xffffffffu;
      }
    } else if (term_abs >= t0) {
      ++rows_seen;
    }
    need_finish = true;
    cursor = seg_end + 1;
  }
  if (bail) {
    if (lane == 0) *reinterpret_cast<volatile uint32_t*>(&P.meta->delta_bail) = 1u;
    return;
  }
  if (lane == 0 && max_line) atomicMax(&P.meta->max_line, max_line);
  if (CF) {
    last_nl_p1 = __reduce_max_sync(0xffffffffu, last_nl_p1);
    if (lane == 0) {
      A.tile_rows[tile] = rows_seen;
      if (last_nl_p1) atomicMax(&P.meta->last_break_p1, last_nl_p1);
      if (rows_seen > A.slot_cap) *reinterpret_cast<volatile uint32_t*>(&P.meta->slot_overflow) = 1u;
    }
  }
}

// Census-free mode, behind pass 1: the rows of tile t start at base[t] (an exclusive scan of tile_rows, whose total is
// meta->tot_rows); the slots go to the global row_rec / row_cnt, and the first malformed row gets its global number.
__global__ void k_row_fixup(const uint32_t* __restrict__ tile_rows, const uint32_t* __restrict__ base, uint32_t ntiles,
                            uint32_t slot_cap, const uint32_t* __restrict__ slot_rec, const uint32_t* __restrict__ slot_cnt,
                            uint32_t* __restrict__ row_rec, uint32_t* __restrict__ row_cnt, EncMeta* __restrict__ meta) {
  if (meta->delta_bail || meta->slot_overflow) return;  // the block is run again: the counts may be incomplete
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0 && meta->bad_slot != ~0ull) meta->bad_row = base[meta->bad_slot >> 32] + (uint32_t)meta->bad_slot;
  const uint64_t tile = i / slot_cap;
  if (tile >= ntiles) return;
  const uint32_t j = (uint32_t)(i - tile * slot_cap);
  if (j < tile_rows[tile]) {
    row_rec[base[tile] + j] = slot_rec[i];
    row_cnt[base[tile] + j] = slot_cnt[i];
  }
}

// Second half of the row-delta pass 1: the value of every listed field (parseInput's strtoull / CHAR tuple /
// Dictionary::insert, ConvertToZDW.cpp:345-402) - p1_process over a flat list, 32 fields a batch, texts parked by
// length class as in k_pass1.  Persistent warps: batch b goes to warp b mod (warps of the grid).
struct D1List {
  const uint32_t* start;
  const uint32_t* len;
  const uint32_t* col;
};
__global__ void __launch_bounds__(ENC_THREADS, 4) k_pass1d_values(const P1Args A, const D1List L, uint32_t rec_cap) {
  __shared__ P1Side s_side[ENC_WARPS][2];
  const EncMeta* meta = A.meta;
  if (meta->delta_bail || meta->rec_overflow) return;
  const unsigned lane = lane_id(), warp = threadIdx.x >> 5;
  const uint32_t total = min(meta->rec_count, rec_cap);
  const uint32_t* wlast = reinterpret_cast<const uint32_t*>(reinterpret_cast<uintptr_t>(A.buf + A.n - 1) & ~(uintptr_t)3);
  P1Side* Q = s_side[warp];
  if (lane < 2) Q[lane].end = Q[lane].done = 0u;
  __syncwarp();
  P1Stats st = {0u, 0u, 0u, 0ull};
  const uint32_t stride = gridDim.x * ENC_WARPS * 32u;
  // one call site: the round after the last batch flushes the parked texts
  for (uint32_t base = (blockIdx.x * ENC_WARPS + warp) * 32u;; base += stride) {
    const bool last = base >= total;
    const uint32_t count = last ? 0u : min(32u, total - base);
    p1_process<1>(A, wlast, L, last ? 0u : base, count, base, nullptr, st, Q, last);
    if (last) break;
  }
  st.max_len = __reduce_max_sync(0xffffffffu, st.max_len);
  st.new_count = __reduce_add_sync(0xffffffffu, st.new_count);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) st.new_bytes += __shfl_xor_sync(0xffffffffu, st.new_bytes, o);
  if (lane == 0 && st.new_count) {
    atomicAdd(&A.meta->n_unique, (unsigned long long)st.new_count);
    atomicAdd(&A.meta->dict_str_bytes, st.new_bytes);
    atomicMax(&A.meta->max_str_len, st.max_len);
  }
}

// ---------------------------------------------------------------------------------------------
// dictionary
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(ENC_THREADS)
    k_ht_compact(const unsigned long long* __restrict__ slots, uint32_t capacity, uint32_t* __restrict__ ustart,
                 uint32_t* __restrict__ ulen, uint32_t* __restrict__ uslot, EncMeta* __restrict__ meta) {
  __shared__ uint32_t ws[34];
  __shared__ uint32_t s_base;
  const uint32_t i = blockIdx.x * ENC_THREADS + threadIdx.x;
  const unsigned long long cur = i < capacity ? slots[i] : 0ull;
  const uint32_t has = cur != 0ull ? 1u : 0u;
  uint32_t total;
  const uint32_t excl = block_exclusive_scan(has, ws, &total);
  if (threadIdx.x == 0) s_base = total ? atomicAdd(&meta->compact_count, total) : 0u;
  __syncthreads();
  if (has) {
    const uint32_t id = s_base + excl;
    ustart[id] = (uint32_t)(cur >> 32) - 1u;
    ulen[id] = (uint32_t)cur;
    uslot[id] = i;
  }
}

__global__ void k_sorted_lens(const uint32_t* __restrict__ order, const uint32_t* __restrict__ ulen, uint32_t n,
                              uint32_t* __restrict__ out) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = ulen[order[i]] + 1u;
}

// dictionary offset of every hash-set slot: offs[i] = sum of (len+1) of the entries sorted before i; offset 0 is the
// origin byte (dictionary.cpp:96-98)
__global__ void k_dict_slots(const uint32_t* __restrict__ order, const uint32_t* __restrict__ uslot,
                             const uint32_t* __restrict__ offs, uint32_t n, uint32_t* __restrict__ slot_off) {
  const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g < n) slot_off[uslot[order[g]]] = 1u + offs[g];
}

// 8 lanes copy one dictionary entry
__global__ void k_dict_emit(const uint8_t* __restrict__ buf, const uint32_t* __restrict__ order,
                            const uint32_t* __restrict__ ustart, const uint32_t* __restrict__ ulen,
                            const uint32_t* __restrict__ offs, uint32_t n, uint8_t* __restrict__ dict_origin) {
  const uint32_t g = (blockIdx.x * blockDim.x + threadIdx.x) >> 3, sub = threadIdx.x & 7;
  if (g >= n) return;
  const uint32_t id = order[g];
  const uint32_t off = 1u + offs[g];
  const uint32_t len = ulen[id];
  const uint8_t* src = buf + ustart[id];
  uint8_t* dst = dict_origin + off;
  for (uint32_t k = sub; k < len; k += 8) dst[k] = __ldg(src + k);
  if (sub == 0) dst[len] = 0;
}

// ---------------------------------------------------------------------------------------------
// column statistics + block header
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(ENC_THREADS)
    k_col_stats(const uint8_t* __restrict__ types, uint32_t ncols, const uint32_t* __restrict__ colset,
                const unsigned long long* __restrict__ colmin, const unsigned long long* __restrict__ colmax,
                uint8_t* __restrict__ csize, unsigned long long* __restrict__ cbase, int32_t* __restrict__ used_idx,
                uint32_t* __restrict__ used_cols, EncMeta* __restrict__ meta) {
  __shared__ uint32_t ws[34];
  __shared__ uint32_t s_sum[ENC_THREADS / 32];
  // Dictionary::getSize() = size + 1; getBytesInOffset(): dictionary.cpp:62-73
  const uint64_t dict_total = meta->dict_str_bytes + 1ull;
  const uint32_t idx_size = bytes_needed(dict_total);
  uint32_t ubase = 0, size_sum = 0;
  for (uint32_t c0 = 0; c0 < ncols; c0 += ENC_THREADS) {
    const uint32_t c = c0 + threadIdx.x;
    uint32_t sz = 0;
    unsigned long long base = 0;
    if (c < ncols && colset[c]) {
      if (is_text_like(types[c])) {
        sz = idx_size;  // every text-like column uses the dictionary's offset width: ConvertToZDW.cpp:447
      } else {
        base = colmin[c] - 1ull;  // :455
        sz = bytes_needed(colmax[c] - base);
      }
    }
    uint32_t total;
    const uint32_t excl = block_exclusive_scan(sz ? 1u : 0u, ws, &total);
    if (c < ncols) {
      csize[c] = (uint8_t)sz;
      cbase[c] = base;
      used_idx[c] = sz ? (int32_t)(ubase + excl) : -1;
      if (sz) used_cols[ubase + excl] = c;
    }
    size_sum += sz;
    ubase += total;
  }
  size_sum = __reduce_add_sync(0xffffffffu, size_sum);
  if ((threadIdx.x & 31) == 0) s_sum[threadIdx.x >> 5] = size_sum;
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t tot = 0;
    for (int w = 0; w < ENC_THREADS / 32; ++w) tot += s_sum[w];
    const uint32_t nflag = (ubase + 7) / 8;
    meta->n_used = ubase;
    meta->nflag = nflag;
    meta->max_row_bytes = nflag + tot;
    meta->idx_size = idx_size;
    meta->dict_total = dict_total;
    if (meta->n_unique == 0ull) {  // empty dictionary: a single 0x00 byte (dictionary.cpp:80-84)
      meta->dict_base = 9;         // (unused)
      meta->stats_base = 10;
    } else {
      meta->dict_base = 9 + 1 + idx_size;  // idxSize byte, totalBytes, then the origin byte
      meta->stats_base = meta->dict_base + dict_total;
    }
    meta->rows_base = meta->stats_base + ncols + 8ull * ubase;
  }
}

__global__ void k_block_header(uint8_t* __restrict__ out, const EncMeta* __restrict__ meta, uint32_t nrows,
                               uint32_t longest_line, uint32_t is_last, uint32_t ncols,
                               const uint8_t* __restrict__ csize, const unsigned long long* __restrict__ cbase,
                               const uint32_t* __restrict__ used_cols) {
  const uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x, nt = gridDim.x * blockDim.x;
  if (tid == 0) {
    for (int k = 0; k < 4; ++k) out[k] = (uint8_t)(nrows >> (8 * k));
    for (int k = 0; k < 4; ++k) out[4 + k] = (uint8_t)(longest_line >> (8 * k));
    out[8] = (uint8_t)is_last;
    if (meta->n_unique == 0ull) {
      out[9] = 0;
    } else {
      out[9] = (uint8_t)meta->idx_size;
      for (uint32_t k = 0; k < meta->idx_size; ++k) out[10 + k] = (uint8_t)(meta->dict_total >> (8 * k));
      out[meta->dict_base] = 0;  // origin byte
    }
  }
  uint8_t* st = out + meta->stats_base;
  for (uint32_t c = tid; c < ncols; c += nt) st[c] = csize[c];
  uint8_t* bs = st + ncols;
  const uint32_t nu = meta->n_used;
  for (uint32_t u = tid; u < nu; u += nt) {
    const unsigned long long b = cbase[used_cols[u]];
    for (int k = 0; k < 8; ++k) bs[(size_t)u * 8 + k] = (uint8_t)(b >> (8 * k));
  }
}

// ---------------------------------------------------------------------------------------------
// pass 2
// ---------------------------------------------------------------------------------------------
// One CTA encodes R consecutive rows from their records.  The values of the rows (and of the row before the first
// one, which the repeat flags of the first row compare against) are scattered into a shared-memory matrix; flags and
// value bytes are then produced row by row, one warp per row.  The tile's bytes go to its own slot of a staging buffer
// (tile * tile_cap); k_gather_tiles packs the tiles once every tile length is known, which keeps the row stream free
// of any cross-CTA dependency while it is being produced.
// what pass 2 needs to know about a column, in one 16-byte load
struct ColInfo {
  unsigned long long base;  // ConvertToZDW.cpp:455 (0 for text-like columns)
  int32_t u;                // index among the used columns, -1 = unused in this block
  uint32_t text;            // the value is a dictionary slot
};
__global__ void k_col_info(const uint8_t* __restrict__ types, const int32_t* __restrict__ used_idx,
                           const unsigned long long* __restrict__ cbase, uint32_t ncols, ColInfo* __restrict__ info) {
  const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= ncols) return;
  ColInfo ci;
  ci.base = cbase[c];
  ci.u = used_idx[c];
  ci.text = is_text_like(types[c]) ? 1u : 0u;
  info[c] = ci;
}

__global__ void __launch_bounds__(ENC_THREADS)
    k_pass2(const uint32_t* __restrict__ rec_col, const unsigned long long* __restrict__ rec_val,
            const uint32_t* __restrict__ row_rec, uint32_t nrows, uint32_t rows_per_cta, const ColInfo* __restrict__ cinfo,
            const uint32_t* __restrict__ slot_off, const uint32_t* __restrict__ used_cols,
            const uint8_t* __restrict__ csize, uint32_t U, uint32_t nflag,
            uint64_t tile_cap, uint8_t* __restrict__ staging, uint64_t* __restrict__ tile_bytes) {
  extern __shared__ __align__(16) uint8_t dsm[];
  // dynamic smem: nval[(R+1)*U] u64 | rowoff[R+1] u32 | rrec[R+2] u32 | usz[U] u8
  unsigned long long* nval = reinterpret_cast<unsigned long long*>(dsm);
  uint32_t* rowoff = reinterpret_cast<uint32_t*>(dsm + (size_t)(rows_per_cta + 1) * U * 8);
  uint32_t* rrec = rowoff + rows_per_cta + 1;
  uint8_t* usz = reinterpret_cast<uint8_t*>(rrec + rows_per_cta + 2);
  const unsigned tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  const uint32_t tile = blockIdx.x;
  const uint32_t r0 = tile * rows_per_cta;
  const uint32_t r1 = min(nrows, r0 + rows_per_cta);
  const uint32_t R = r1 - r0;
  const uint32_t rw0 = r0 ? r0 - 1 : 0;     // first row whose records are needed
  const uint32_t nrw = r1 - rw0;             // rows loaded
  for (uint32_t k = tid; k < (R + 1) * U; k += ENC_THREADS) nval[k] = 0ull;
  for (uint32_t u = tid; u < U; u += ENC_THREADS) usz[u] = csize[used_cols[u]];
  for (uint32_t k = tid; k <= nrw; k += ENC_THREADS) rrec[k] = row_rec[rw0 + k];
  __syncthreads();

  // ---- values of the tile's rows and of the row before it, from the records; four records per thread and round, so
  // that the dependent loads (record -> column info -> dictionary offset) of different records overlap
  {
    const uint32_t k0 = rrec[0], k1 = rrec[nrw];
    constexpr int NR = 4;
    for (uint32_t kb = k0 + tid; kb < k1; kb += NR * ENC_THREADS) {
      uint32_t col[NR];
      unsigned long long v[NR];
      ColInfo ci[NR];
#pragma unroll
      for (int j = 0; j < NR; ++j) {
        const uint32_t k = kb + (uint32_t)j * ENC_THREADS;
        col[j] = k < k1 ? rec_col[k] : REC_EMPTY;
        v[j] = k < k1 ? rec_val[k] : 0ull;
      }
#pragma unroll
      for (int j = 0; j < NR; ++j) {
        ci[j].u = -1;
        ci[j].text = 0;
        ci[j].base = 0;
        if (col[j] != REC_EMPTY) {
          const uint4 q = __ldg(reinterpret_cast<const uint4*>(cinfo + col[j]));
          ci[j].base = (unsigned long long)q.x | ((unsigned long long)q.y << 32);
          ci[j].u = (int32_t)q.z;
          ci[j].text = q.w;
        }
      }
#pragma unroll
      for (int j = 0; j < NR; ++j) {
        if (ci[j].u < 0) continue;
        if (ci[j].text) v[j] = __ldg(slot_off + (uint32_t)v[j]);  // Dictionary::getOffset
        else if (v[j]) v[j] -= ci[j].base;                        // ConvertToZDW.cpp:548,566
      }
#pragma unroll
      for (int j = 0; j < NR; ++j) {
        if (ci[j].u < 0) continue;
        const uint32_t k = kb + (uint32_t)j * ENC_THREADS;
        // row of the record: last a with rrec[a] <= k
        uint32_t a = 0, b = nrw;
        while (b - a > 1) {
          const uint32_t m = (a + b) >> 1;
          if (rrec[m] <= k) a = m;
          else b = m;
        }
        nval[(size_t)(rw0 + a + 1 - r0) * U + (uint32_t)ci[j].u] = v[j];
      }
    }
  }
  __syncthreads();

  // ---- encoded length of every row: nflag + sum of the sizes of the changed columns
  for (uint32_t j = warp; j < R; j += ENC_WARPS) {
    const unsigned long long* cur = nval + (size_t)(j + 1) * U;
    const unsigned long long* prv = nval + (size_t)j * U;
    uint32_t acc = 0;
    for (uint32_t u = lane; u < U; u += 32)
      if (cur[u] != prv[u]) acc += usz[u];
    acc = __reduce_add_sync(0xffffffffu, acc);
    if (lane == 0) rowoff[j] = nflag + acc;
  }
  __syncthreads();
  // exclusive scan of the row lengths (R is small; warp 0 walks it in chunks of 32)
  if (warp == 0) {
    uint32_t run = 0;
    for (uint32_t j0 = 0; j0 < R; j0 += 32) {
      const uint32_t j = j0 + lane;
      const uint32_t v = j < R ? rowoff[j] : 0u;
      uint32_t inc = v;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= (unsigned)o) inc += t;
      }
      if (j < R) rowoff[j] = run + inc - v;
      run += __shfl_sync(0xffffffffu, inc, 31);
    }
    if (lane == 0) {
      rowoff[R] = run;
      tile_bytes[tile] = run;
    }
  }
  __syncthreads();
  uint8_t* tile_out = staging + (uint64_t)tile * tile_cap;

  // ---- emit: flag bytes, then the low columnSize bytes of every changed value (little-endian)
  for (uint32_t j = warp; j < R; j += ENC_WARPS) {
    const unsigned long long* cur = nval + (size_t)(j + 1) * U;
    const unsigned long long* prv = nval + (size_t)j * U;
    uint8_t* orow = tile_out + rowoff[j];
    uint32_t voff = nflag;
    for (uint32_t ub = 0; ub < U; ub += 32) {
      const uint32_t u = ub + lane;
      unsigned long long v = 0;
      bool flag = false;
      if (u < U) {
        v = cur[u];
        flag = v != prv[u];
      }
      const unsigned bal = __ballot_sync(0xffffffffu, flag);
      if (lane < 4 && (ub >> 3) + lane < nflag) orow[(ub >> 3) + lane] = (uint8_t)(bal >> (8 * lane));
      const uint32_t sz = flag ? usz[u] : 0u;
      uint32_t inc = sz;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= (unsigned)o) inc += t;
      }
      const uint32_t tot = __shfl_sync(0xffffffffu, inc, 31);
      if (flag) {
        uint8_t* d = orow + voff + inc - sz;
        for (uint32_t b = 0; b < sz; ++b) d[b] = (uint8_t)(v >> (8 * b));
      }
      voff += tot;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// pass 2, row-delta variant: the records of a row are exactly the columns whose field changed against the row before,
// and k_pass1d_values has already decided for each whether the VALUE changed (rec_col without REC_SAME: the reference's
// flag, ConvertToZDW.cpp:532,548,567).  A row's bytes therefore follow from its own records: k_p2d_rowlen sums the
// sizes of the flagged columns (before pass 1's read-back, so the exact output size comes back with it), k_p2d_emit
// writes flags and value bytes straight to the row's place in the output.  A row's records are two runs in column
// order - the "became empty" ones, then the changed fields - and every value goes behind the sizes of the records of
// both runs with a smaller column.
// ---------------------------------------------------------------------------------------------
// value a record stands for in the row stream: dictionary offset / number minus the column's base (0 stays 0)
__device__ __forceinline__ unsigned long long record_value(const ColInfo& ci, const uint32_t* __restrict__ slot_off,
                                                           unsigned long long v) {
  if (v == 0ull) return 0ull;
  return ci.text ? (unsigned long long)__ldg(slot_off + (uint32_t)(v - 1ull)) : v - ci.base;  // :548,566; Dictionary::getOffset
}

// one warp per row: row_off[r] = nflag + the sizes of the flagged records' columns (csize is 0 for a column the block
// does not use).  rows_cap rows are written, those at or past the block's row count with 0, so that an exclusive scan
// over all of them gives the row offsets and the total; census-free, the row count is only known on the device.
__global__ void __launch_bounds__(ENC_THREADS)
    k_p2d_rowlen(const uint32_t* __restrict__ rec_col, const uint32_t* __restrict__ row_rec, const uint32_t* __restrict__ row_cnt,
                 uint32_t rows_cap, bool census_free, const uint8_t* __restrict__ csize, const EncMeta* __restrict__ meta,
                 uint64_t* __restrict__ row_off) {
  // Pass 1 runs again, or the general one: row_off stays unwritten, and the scan behind this kernel leaves a
  // meaningless meta->rows_bytes, which the host reads only from a run of pass 1 that went through
  if (meta->delta_bail || meta->rec_overflow || meta->slot_overflow) return;
  const unsigned lane = lane_id();
  const uint32_t nrows = census_free ? min(meta->tot_rows, rows_cap) : rows_cap, nflag = meta->nflag;
  for (uint32_t r = blockIdx.x * ENC_WARPS + (threadIdx.x >> 5); r < rows_cap; r += gridDim.x * ENC_WARPS) {
    uint32_t acc = 0;
    if (r < nrows) {
      const uint32_t k0 = row_rec[r], cnt = row_cnt[r] & 0xffffu;
      for (uint32_t i = lane; i < cnt; i += 32u) {
        const uint32_t c = rec_col[k0 + i];
        if (!(c & REC_SAME)) acc += csize[c];
      }
      acc = nflag + __reduce_add_sync(0xffffffffu, acc);
    }
    if (lane == 0) row_off[r] = acc;
  }
}

struct P2DWarp {                // (16-bit prefixes: a row's value bytes are at most 2 * DCAP * 8; 8 CTAs fit an SM)
  uint16_t col[2 * DCAP];      // the row's records: column
  uint16_t pre[2 * DCAP + 1];  // ... value bytes of the records in front of it (record order)
  uint32_t flags[DBW];         // the row's flag bytes: bit u = used column u
};

__global__ void __launch_bounds__(ENC_THREADS)
    k_p2d_emit(const uint32_t* __restrict__ rec_col, const unsigned long long* __restrict__ rec_val,
               const uint32_t* __restrict__ row_rec, const uint32_t* __restrict__ row_cnt, const uint64_t* __restrict__ row_off,
               uint32_t nrows, uint32_t nflag, const ColInfo* __restrict__ cinfo, const uint8_t* __restrict__ csize,
               const uint32_t* __restrict__ slot_off, uint8_t* __restrict__ rows_out) {
  __shared__ P2DWarp sw[ENC_WARPS];
  const unsigned lane = lane_id();
  P2DWarp& W = sw[threadIdx.x >> 5];
  const uint32_t nfw = (nflag + 3u) >> 2;
  for (uint32_t r = blockIdx.x * ENC_WARPS + (threadIdx.x >> 5); r < nrows; r += gridDim.x * ENC_WARPS) {
    const uint32_t k0 = row_rec[r], cw = row_cnt[r], cnt = cw & 0xffffu, nte = cw >> 16;
    uint8_t* orow = rows_out + row_off[r];
    for (uint32_t w = lane; w < nfw; w += 32u) W.flags[w] = 0u;
    __syncwarp();
    // ---- columns, value sizes and flags of the records
    uint32_t run = 0;
    for (uint32_t i0 = 0; i0 < cnt; i0 += 32u) {
      const uint32_t i = i0 + lane;
      uint32_t sz = 0;
      if (i < cnt) {
        const uint32_t c = rec_col[k0 + i], col = c & ~REC_SAME;
        W.col[i] = (uint16_t)col;
        if (!(c & REC_SAME)) {
          sz = csize[col];
          if (sz) {
            const uint32_t u = (uint32_t)__ldg(&cinfo[col].u);
            atomicOr(&W.flags[u >> 5], 1u << (u & 31u));
          }
        }
      }
      uint32_t inc = sz;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= (unsigned)o) inc += t;
      }
      if (i < cnt) W.pre[i] = (uint16_t)(run + inc - sz);
      run += __shfl_sync(0xffffffffu, inc, 31);
    }
    if (lane == 0) W.pre[cnt] = (uint16_t)run;
    __syncwarp();
    for (uint32_t b = lane; b < nflag; b += 32u) orow[b] = (uint8_t)(W.flags[b >> 2] >> (8u * (b & 3u)));
    // ---- value bytes (low csize bytes, little-endian): behind the flagged records of its own run in front of it and
    // those of the other run with a smaller column (a column is in at most one of the runs)
    for (uint32_t i = lane; i < cnt; i += 32u) {
      const uint32_t sz = (uint32_t)W.pre[i + 1] - W.pre[i];
      if (!sz) continue;
      const uint32_t col = W.col[i];
      const bool first = i < nte;
      const uint32_t ob = first ? nte : 0u, oe = first ? cnt : nte;
      uint32_t lo = ob, hi = oe;  // first record of the other run whose column is not smaller
      while (lo < hi) {
        const uint32_t m = (lo + hi) >> 1;
        if (W.col[m] < col) lo = m + 1;
        else hi = m;
      }
      const uint32_t own = first ? (uint32_t)W.pre[i] : (uint32_t)W.pre[i] - W.pre[nte];
      const uint4 q = __ldg(reinterpret_cast<const uint4*>(cinfo + col));
      ColInfo ci;
      ci.base = (unsigned long long)q.x | ((unsigned long long)q.y << 32);
      ci.u = (int32_t)q.z;
      ci.text = q.w;
      const unsigned long long v = record_value(ci, slot_off, rec_val[k0 + i]);
      uint8_t* d = orow + nflag + own + ((uint32_t)W.pre[lo] - W.pre[ob]);
      for (uint32_t b = 0; b < sz; ++b) d[b] = (uint8_t)(v >> (8u * b));
    }
    __syncwarp();  // the next row refills the lists
  }
}

// Little-endian 32-bit words of the byte string that starts at an arbitrary address: aligned loads + funnel shift.
struct WordStream {
  const uint32_t* w;
  uint32_t sh, cur;
  __device__ __forceinline__ explicit WordStream(const uint8_t* a) {
    const uintptr_t u = reinterpret_cast<uintptr_t>(a);
    w = reinterpret_cast<const uint32_t*>(u & ~(uintptr_t)3);
    sh = (uint32_t)(u & 3u) * 8u;
    cur = __ldg(w);
  }
  __device__ __forceinline__ uint32_t next() {
    const uint32_t nx = __ldg(++w);
    const uint32_t r = __funnelshift_r(cur, nx, sh);
    cur = nx;
    return r;
  }
};

// packs the staged tiles into the row stream: tile t's bytes go to out_rows + tile_off[t]
__global__ void __launch_bounds__(ENC_THREADS)
    k_gather_tiles(const uint8_t* __restrict__ staging, uint64_t tile_cap, const uint64_t* __restrict__ tile_off,
                   const uint64_t* __restrict__ tile_bytes, uint8_t* __restrict__ out_rows) {
  const uint32_t tile = blockIdx.x;
  const uint8_t* src = staging + (uint64_t)tile * tile_cap;
  uint8_t* dst = out_rows + tile_off[tile];
  const uint32_t nb = (uint32_t)tile_bytes[tile];
  // head bytes up to a 16-byte aligned destination, 16-byte body through a funnel of source words, byte tail
  const uint32_t head = min(nb, (uint32_t)((16u - (uint32_t)(reinterpret_cast<uintptr_t>(dst) & 15u)) & 15u));
  for (uint32_t k = threadIdx.x; k < head; k += ENC_THREADS) dst[k] = src[k];
  const uint32_t body = (nb - head) >> 4;
  for (uint32_t q = threadIdx.x; q < body; q += ENC_THREADS) {
    const uint8_t* s = src + head + (size_t)q * 16;
    WordStream ws(s);
    uint4 v;
    v.x = ws.next();
    v.y = ws.next();
    v.z = ws.next();
    v.w = ws.next();
    *reinterpret_cast<uint4*>(dst + head + (size_t)q * 16) = v;
  }
  for (uint32_t k = head + body * 16 + threadIdx.x; k < nb; k += ENC_THREADS) dst[k] = src[k];
}

__global__ void k_init_minmax(unsigned long long* colmin, unsigned long long* colmax, uint32_t* colset, uint32_t ncols) {
  uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < ncols) {
    colmin[c] = ~0ull;
    colmax[c] = 0ull;
    colset[c] = 0u;
  }
}

// ---------------------------------------------------------------------------------------------
// where would the reference close the block?  (opts.heap_blocks = K, SURVEY 8f-1 / App. B-14)
//
// The reference copies every NEW string into 64 MiB string-heap blocks in the order it meets them - row by row, column by
// column - and ends the ZDW block on the insert that opens heap block K (stringheap.cpp:31-59,75-86; ConvertToZDW.cpp
// :334-355,404-413).  After the general pass 1 the records of the buffer are in exactly that order and a text record
// holds its string's hash-set slot, so: the first record of every slot is the string's first occurrence
// (k_heap_first_ord), its length + 1 the bytes it takes on the heap (k_heap_new_len), a prefix sum over the records
// the heap's fill level, and K - 1 binary searches over that prefix find the record whose string does not fit the
// current heap block any more (k_heap_cut).
// ---------------------------------------------------------------------------------------------
struct HeapCut {
  uint32_t found;     // heap block K was opened inside the buffer
  uint32_t row;       // rows in front of the row whose insert opened it (= rows of the block)
  uint32_t col;       // column of that insert
  uint32_t allocs;    // heap blocks opened in the whole buffer (when !found)
};

__global__ void k_heap_first_ord(const uint32_t* __restrict__ rec_col, const unsigned long long* __restrict__ rec_val,
                                 const uint8_t* __restrict__ types, uint32_t nrec, uint32_t* __restrict__ first_ord) {
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= nrec) return;
  const uint32_t col = rec_col[k];
  if (col == REC_EMPTY || !is_text_like(__ldg(types + col))) return;
  atomicMin(&first_ord[(uint32_t)rec_val[k]], k);
}
__global__ void k_heap_new_len(const uint32_t* __restrict__ rec_col, const unsigned long long* __restrict__ rec_val,
                               const uint8_t* __restrict__ types, uint32_t nrec, const uint32_t* __restrict__ first_ord,
                               const unsigned long long* __restrict__ slots, uint64_t* __restrict__ new_len) {
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= nrec) return;
  const uint32_t col = rec_col[k];
  uint64_t v = 0;
  if (col != REC_EMPTY && is_text_like(__ldg(types + col))) {
    const uint32_t slot = (uint32_t)rec_val[k];
    if (first_ord[slot] == k) v = (uint64_t)(uint32_t)slots[slot] + 1ull;  // strlen + 1, StringHeap::copyToHeap
  }
  new_len[k] = v;
}
// one thread: pre[k] = heap bytes of the new strings in front of record k, len[k] = bytes of record k's string if new
__global__ void k_heap_cut(const uint64_t* __restrict__ pre, const uint64_t* __restrict__ len, uint32_t nrec, uint64_t total,
                           uint32_t K, const uint32_t* __restrict__ row_rec, uint32_t nrows, const uint32_t* __restrict__ rec_col,
                           HeapCut* __restrict__ out) {
  const uint64_t HEAP_BLOCK = 64ull << 20;
  out->found = 0;
  out->row = out->col = 0;
  uint32_t allocs = 0, at = 0;
  uint64_t limit = 0;  // the heap is full once the bytes up to and including a new string exceed this
  bool have = false;
  for (;;) {
    // first record k >= at whose new string ends behind `limit` (pre + len is non-decreasing and only grows at new strings)
    uint32_t a = at, b = nrec;
    while (a < b) {
      const uint32_t m = a + ((b - a) >> 1);
      const uint64_t end = pre[m] + len[m];
      if (have ? end > limit : end > 0) b = m;
      else a = m + 1;
    }
    if (a >= nrec) break;  // everything else fits
    ++allocs;
    if (allocs >= K) {
      // row of record a: last r with row_rec[r] <= a
      uint32_t lo = 0, hi = nrows;
      while (hi - lo > 1) {
        const uint32_t m = (lo + hi) >> 1;
        if (row_rec[m] <= a) lo = m;
        else hi = m;
      }
      out->found = 1;
      out->row = lo;
      out->col = rec_col[a];
      break;
    }
    const uint64_t l = len[a];
    limit = pre[a] + (l > HEAP_BLOCK ? l : HEAP_BLOCK);  // the new heap block starts with this string
    have = true;
    at = a + 1;
  }
  out->allocs = allocs;
  (void)total;
}

uint32_t longest_line_field(uint32_t prev, uint32_t max_line) {
  // smallest 16384 * 2^k >= L + 1, cumulative over the file (getnextrow.cpp:57-65; SURVEY App. B-13)
  uint64_t cap = prev ? prev : 16384u;
  while (cap < (uint64_t)max_line + 1ull) cap *= 2;
  return (uint32_t)cap;
}

}  // namespace

// =================================================================================================
// host driver
// =================================================================================================
namespace {
struct HeapProbe {  // the probe run of opts.heap_blocks: K in, the cut out
  uint32_t K;
  bool found;
  uint32_t row, col, allocs;
};
}  // namespace

static int encode_block_run(Ctx* ctx, const zdwb_schema* schema, const void* tsv, size_t n, const zdwb_encode_opts* opts,
                            zdwb_block_out* out, HeapProbe* probe);

int encode_block_impl(Ctx* ctx, const zdwb_schema* schema, const void* tsv, size_t n, const zdwb_encode_opts* opts,
                      zdwb_block_out* out) {
  if (!opts->heap_blocks || opts->max_rows) return encode_block_run(ctx, schema, tsv, n, opts, out, nullptr);
  // ---- the reference's own cut: a probe run of pass 1 over the whole buffer finds the insert that opens heap block K,
  // the block is then encoded with the (rows, spilled columns) that follow from it.  The buffer is made resident first:
  // both runs read it.
  memset(out, 0, sizeof(*out));
  if (n == 0 || n >= 0xffffff00ull) return encode_block_run(ctx, schema, tsv, n, opts, out, nullptr);
  void* resident = nullptr;
  zdwb_encode_opts o = *opts;
  const void* src = tsv;
  if (!opts->input_on_device) {
    if (cudaMalloc(&resident, n + 64) != cudaSuccess) {
      (void)cudaGetLastError();
      ctx->err = "encode: device allocation of the input window failed";
      return ZDWB_ERR_OOM;
    }
    if (cudaMemcpyAsync(resident, tsv, n, cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess ||
        cudaStreamSynchronize(ctx->stream) != cudaSuccess) {
      (void)cudaGetLastError();
      cudaFree(resident);
      ctx->err = "encode: copy of the input window failed";
      return ZDWB_ERR_CUDA;
    }
    src = resident;
    o.input_on_device = 1;
  }
  HeapProbe probe = {opts->heap_blocks, false, 0, 0, 0};
  zdwb_encode_opts po = o;
  po.heap_blocks = 0;
  po.output_on_device = 1;
  int rc = encode_block_run(ctx, schema, src, n, &po, out, &probe);
  if (rc == ZDWB_OK && out->rows_in_buffer) {
    zdwb_encode_opts fo = o;
    fo.heap_blocks = 0;
    if (probe.found && probe.row == 0) {
      ctx->err = "encode: string heap block " + std::to_string(opts->heap_blocks) + " opens inside the first row (the reference's OUT_OF_MEMORY)";
      rc = ZDWB_ERR_OOM;  // ConvertToZDW.cpp:824-834
    } else if (probe.found) {
      fo.max_rows = probe.row;
      fo.spill_cols = probe.col + 1;
      rc = encode_block_run(ctx, schema, src, n, &fo, out, nullptr);
    } else if (opts->more_input_follows) {
      // the heap block does not open inside this window: the caller widens it (nothing is consumed)
      const uint64_t rows = out->rows_in_buffer;
      memset(out, 0, sizeof(*out));
      out->rows_in_buffer = rows;
    } else {
      rc = encode_block_run(ctx, schema, src, n, &fo, out, nullptr);
    }
  }
  if (resident) {
    cudaStreamSynchronize(ctx->stream);
    cudaFree(resident);
  }
  return rc;
}

static int encode_block_run(Ctx* ctx, const zdwb_schema* schema, const void* tsv, size_t n, const zdwb_encode_opts* opts,
                            zdwb_block_out* out, HeapProbe* probe) {
  memset(out, 0, sizeof(*out));
  ZDWB_TRY(call_begin(ctx));
  cudaStream_t st = ctx->stream;
  const uint32_t ncols = schema->ncols;
  if (ncols == 0 || !schema->types) {
    ctx->err = "encode: schema has no columns";
    return ZDWB_ERR_BAD_ARG;
  }
  for (uint32_t c = 0; c < ncols; ++c) {
    if (!is_known_type(schema->types[c])) {
      ctx->err = "encode: unsupported column type id " + std::to_string((int)schema->types[c]);
      return ZDWB_ERR_UNSUPPORTED;
    }
  }
  if (n >= 0xffffff00ull) {
    ctx->err = "encode: a block's TSV must be smaller than 4 GiB (row offsets are 32-bit); split the input";
    return ZDWB_ERR_UNSUPPORTED;
  }
  if (n == 0) return ZDWB_OK;

  // ---- input residency
  DevBuf tsv_dev;
  const uint8_t* buf;
  if (opts->input_on_device) {
    buf = static_cast<const uint8_t*>(tsv);
  } else {
    ZDWB_TRY(tsv_dev.alloc(ctx, n + 64));
    if (n >= ((size_t)32 << 20) && is_pageable_host(tsv)) {
      // pageable caller memory: through the pinned ring, chunk by chunk (the driver's own staging is several times slower)
      const uint8_t* src = static_cast<const uint8_t*>(tsv);
      ZDWB_TRY(ring_h2d(ctx, tsv_dev.p, n, [src](void* dst, size_t off, size_t k) {
        memcpy(dst, src + off, k);
        return true;
      }));
    } else if (ctx->copy_gate && n >= COPY_GATE_MIN) {
      std::lock_guard<std::mutex> turn(copy_gate(ctx->device, 0));
      ZDWB_CUDA_TRY(ctx, cudaMemcpyAsync(tsv_dev.p, tsv, n, cudaMemcpyHostToDevice, st));
      ZDWB_CUDA_TRY(ctx, cudaStreamSynchronize(st));
    } else {
      ZDWB_CUDA_TRY(ctx, cudaMemcpyAsync(tsv_dev.p, tsv, n, cudaMemcpyHostToDevice, st));
    }
    buf = tsv_dev.as<uint8_t>();
  }
  const int64_t lo = -(int64_t)(reinterpret_cast<uintptr_t>(buf) & 15u);

  DevBuf meta_d, types_d;
  ZDWB_TRY(meta_d.alloc(ctx, sizeof(EncMeta)));
  ZDWB_TRY(types_d.alloc(ctx, ncols));
  EncMeta* meta = meta_d.as<EncMeta>();
  EncMeta* hmeta = static_cast<EncMeta*>(ctx->meta_host);
  auto reset_meta = [&]() -> int {
    ZDWB_CUDA_TRY(ctx, cudaMemsetAsync(meta, 0, sizeof(EncMeta), st));
    ZDWB_CUDA_TRY(ctx, cudaMemsetAsync(&meta->bad_row, 0xff, 4, st));  // 0xffffffff = no malformed row
    ZDWB_CUDA_TRY(ctx, cudaMemsetAsync(&meta->bad_slot, 0xff, 8, st));
    return ZDWB_OK;
  };
  ZDWB_TRY(reset_meta());
  {
    void* pinned = stage_take(ctx, ncols);
    if (!pinned) {
      ctx->err = "encode: pinned staging allocation failed";
      return ZDWB_ERR_OOM;
    }
    memcpy(pinned, schema->types, ncols);
    ZDWB_CUDA_TRY(ctx, cudaMemcpyAsync(types_d.p, pinned, ncols, cudaMemcpyHostToDevice, st));
  }

  // ---- which pass 1?  The row-delta variant (k_pass1d) pays on wide rows; narrow rows - and rows that do not fit its
  // per-warp lists - go through the general one (k_pass1).  Both leave records for their own pass 2.
  const uint64_t DELTA_MIN_ROW_BYTES = 512;
  bool delta = !probe && ctx->enc_delta != 0 && ncols <= DELTA_MAX_COLS && n >= 64 &&
               (ctx->enc_delta == 1 || (!ctx->delta_bailed && (ctx->last_row_bytes == 0 || ctx->last_row_bytes >= DELTA_MIN_ROW_BYTES)));
  // A delta block that is not cut (max_rows) can do without the row census: pass 1 finds every tile's reference row
  // itself and numbers the tile's rows from 0 (k_pass1d<true>, then k_row_fixup), which saves a read of the TSV and a
  // host round trip.  Automatic once a delta block of this context has shown how wide the rows are; the first block of
  // a context, cut blocks and blocks whose tiles hold more rows than they have slots for take the census (and after such
// a fall-back, the context's later blocks).
  bool census_free = delta && opts->max_rows == 0 &&
                     (ctx->enc_census == 0 || (ctx->enc_census < 0 && ctx->last_row_bytes >= DELTA_MIN_ROW_BYTES &&
                                               !ctx->delta_bailed && ctx->last_records && !ctx->census_fell_back));

  DevBuf agg, colset, colmin, colmax, slots, rec_col, rec_val, row_rec, row_cnt, chg_start, chg_len, csize, cbase, used_idx, used_cols;
  DevBuf slot_rec, slot_cnt, tile_rows, tile_base, row_off;
  HashTable ht{nullptr, 0};
  uint32_t nrows = 0;
  bool is_last = false;
  uint32_t spill_row_len = 0, tail_bytes = 0;
  uint64_t rows_total = 0, ne_total = 0;
  for (;;) {  // the census-free run may hand the block to the census, the delta variant to the general one
    // ---- census: per-tile counts and their prefix
    // (delta: a warp walks its tile row by row, so a small input is cut into smaller tiles - down to 8 KiB - until there
    // are about as many as warps fit on the GPU; every tile re-reads the row in front of it, which is why not smaller)
    uint32_t tile_bytes = TILE;
    if (delta) {
      tile_bytes = DTILE;
      while (tile_bytes > 8192 && ((uint64_t)(-lo) + n) / tile_bytes < (uint64_t)ctx->sm_count * 32) tile_bytes >>= 1;
      if (ctx->enc_dtile >= 2048 && ctx->enc_dtile <= (1 << 20) && (ctx->enc_dtile & (ctx->enc_dtile - 1)) == 0)
        tile_bytes = (uint32_t)ctx->enc_dtile;
    }
    const uint64_t span = (uint64_t)(-lo) + n;
    const uint32_t ntiles = (uint32_t)((span + tile_bytes - 1) / tile_bytes);
    const uint32_t tile_ctas = (ntiles + ENC_WARPS - 1) / ENC_WARPS;
    // census-free: row slots per tile.  A valid row is at least ncols bytes (its tabs and terminator), so
    // ceil(tile / ncols) always suffice; in automatic mode a quarter of the previous block's mean row bounds them for
    // narrow schemas
    uint32_t slot_cap = 0;
    if (census_free) {
      const uint64_t min_row = std::max<uint64_t>({(uint64_t)ncols, 2, ctx->enc_census < 0 ? ctx->last_row_bytes / 4 : 0});
      slot_cap = (uint32_t)((tile_bytes + min_row - 1) / min_row);
      if ((uint64_t)ntiles * slot_cap > (n >> 3) + (1u << 20)) census_free = false;  // too many slots: take the census
    }
    uint64_t limit = n;  // bytes that belong to the block (census-free: pass 1 drops a row the buffer's end cuts short)
    // The block's rows and extent from the window's totals in hmeta (census: before pass 1; census-free: after it, and
    // never cut).  *next: 0 = go on, 1 = the window holds no complete row, 2 = narrow rows: the general variant.
    auto settle = [&](int* next) -> int {
      *next = 0;
      rows_total = hmeta->tot_rows;
      const uint64_t tail_start = hmeta->last_break_p1;  // first byte after the last row break
      out->rows_in_buffer = rows_total;
      if (rows_total == 0) {
        out->tsv_consumed = opts->more_input_follows ? 0 : n;  // a window without a complete row: the caller widens it
        *next = 1;
        return ZDWB_OK;  // "Empty data file -- nothing to process", ConvertToZDW.cpp:824-835
      }
      ctx->last_row_bytes = std::max<uint64_t>(1, tail_start / rows_total);
      if (delta && ctx->enc_delta != 1 && ctx->last_row_bytes < DELTA_MIN_ROW_BYTES) {
        *next = 2;  // narrow rows: the general pass 1 (and its census)
        return ZDWB_OK;
      }

      const uint64_t nrows64 = (opts->max_rows && opts->max_rows < rows_total) ? opts->max_rows : rows_total;
      nrows = (uint32_t)nrows64;
      const bool took_all = nrows64 == rows_total;
      is_last = took_all && !opts->more_input_follows;

      // ---- block extent
      spill_row_len = 0;  // the interrupted row was read in full before it was dropped: it counts for longestLine
      tail_bytes = 0;
      if (took_all) {
        // the terminator of the last row is the last row break unless blank lines follow it; either way every
        // delimiter in front of tail_start belongs to the block
        limit = tail_start;
        if (is_last) {
          out->tsv_consumed = n;
          tail_bytes = (uint32_t)(n - tail_start);
        } else {
          out->tsv_consumed = tail_start;  // the unterminated tail belongs to the next window
        }
      } else {
        ZDWB_TRY(launch(ctx, "k_find_cut", k_find_cut, 1, 32, 0, buf, n, lo, ntiles, tile_bytes, agg.as<TileAgg>(), nrows - 1, meta));
        ZDWB_CUDA_TRY(ctx, cudaMemcpyAsync(hmeta, meta, sizeof(EncMeta), cudaMemcpyDeviceToHost, st));
        ZDWB_CUDA_TRY(ctx, cudaStreamSynchronize(st));
        limit = hmeta->cut_end_p1;
        out->tsv_consumed = hmeta->next_start;
        {
          // the row behind the block has been read in full when the block is closed - the row buffer has grown with it
          // (getnextrow.cpp:57-65), so its length counts for longestLine - and its first spill_cols columns have been parsed
          ZDWB_TRY(launch(ctx, "k_find_spill", k_find_spill, 1, 1, 0, buf, n, hmeta->next_start, opts->spill_cols, meta));
          ZDWB_CUDA_TRY(ctx, cudaMemcpyAsync(hmeta, meta, sizeof(EncMeta), cudaMemcpyDeviceToHost, st));
          ZDWB_CUDA_TRY(ctx, cudaStreamSynchronize(st));
          if (hmeta->spill_row_len) {
            if (opts->spill_cols) limit = hmeta->spill_end;  // pass 1 takes every field whose closing delimiter lies in front of this
            spill_row_len = hmeta->spill_row_len;
          }
        }
      }
      out->nrows = nrows;
      return ZDWB_OK;
    };
    if (!census_free) {
      ZDWB_TRY(agg.alloc(ctx, (size_t)ntiles * sizeof(TileAgg)));
      if (delta)
        ZDWB_TRY(launch(ctx, "k_row_census", k_row_census, tile_ctas, ENC_THREADS, 0, buf, n, lo, ntiles, tile_bytes, agg.as<TileAgg>()));
      else
        ZDWB_TRY(launch(ctx, "k_tile_count", k_tile_count, tile_ctas, ENC_THREADS, 0, buf, n, lo, ntiles, agg.as<TileAgg>()));
      {
        const uint32_t nparts = (ntiles + TS_THREADS - 1) / TS_THREADS;
        DevBuf part;
        ZDWB_TRY(part.alloc(ctx, (size_t)nparts * sizeof(TileAgg)));
        ZDWB_TRY(launch(ctx, "k_tile_scan", k_tile_scan_local, nparts, TS_THREADS, 0, agg.as<TileAgg>(), ntiles, part.as<TileAgg>()));
        ZDWB_TRY(launch(ctx, "k_tile_scan", k_tile_scan, 1, TS_THREADS, 0, part.as<TileAgg>(), nparts, meta));
        ZDWB_TRY(launch(ctx, "k_tile_scan", k_tile_scan_add, nparts, TS_THREADS, 0, agg.as<TileAgg>(), ntiles, part.as<TileAgg>()));
      }
      ZDWB_CUDA_TRY(ctx, cudaMemcpyAsync(hmeta, meta, sizeof(EncMeta), cudaMemcpyDeviceToHost, st));
      ZDWB_CUDA_TRY(ctx, cudaStreamSynchronize(st));
      int next;
      ZDWB_TRY(settle(&next));
      if (next == 1) return ZDWB_OK;
      if (next == 2) {
        delta = false;
        continue;
      }
    }

    // ---- pass 1 (retry with a larger hash set / larger record arrays when they fill up)
    ZDWB_TRY(colset.alloc(ctx, (size_t)ncols * 4));
    ZDWB_TRY(colmin.alloc(ctx, (size_t)ncols * 8));
    ZDWB_TRY(colmax.alloc(ctx, (size_t)ncols * 8));
    ZDWB_TRY(csize.alloc(ctx, ncols));
    ZDWB_TRY(cbase.alloc(ctx, (size_t)ncols * 8));
    ZDWB_TRY(used_idx.alloc(ctx, (size_t)ncols * 4));
    ZDWB_TRY(used_cols.alloc(ctx, (size_t)ncols * 4));
    ne_total = hmeta->tot_ne;  // (general variant only: the delta census does not count fields)
    uint64_t rec_cap = 0;
    const uint64_t nslots = (uint64_t)ntiles * slot_cap;
    const uint64_t rows_cap = census_free ? nslots : nrows;  // (delta: rows pass 1 can number)
    if (delta) {
      // a row's records = its changed fields + the columns that became empty; sized from the previous block of the
      // file (blocks look alike) or from the bytes, and grown on overflow
      rec_cap = std::max<uint64_t>({ctx->last_records + ctx->last_records / 2, limit / 16, (uint64_t)1 << 16});
      rec_cap = std::min<uint64_t>(rec_cap, limit + 64);
      ZDWB_TRY(row_rec.alloc(ctx, (size_t)(rows_cap + 2) * 4));
      ZDWB_TRY(row_cnt.alloc(ctx, (size_t)(rows_cap + 2) * 4));
      ZDWB_TRY(row_off.alloc(ctx, (size_t)(rows_cap + 2) * 8));
      if (census_free) {
        ZDWB_TRY(slot_rec.alloc(ctx, (size_t)nslots * 4));
        ZDWB_TRY(slot_cnt.alloc(ctx, (size_t)nslots * 4));
        ZDWB_TRY(tile_rows.alloc(ctx, (size_t)ntiles * 4));
        ZDWB_TRY(tile_base.alloc(ctx, (size_t)ntiles * 4));
      }
    } else {
      rec_cap = ne_total;
      ZDWB_TRY(row_rec.alloc(ctx, (size_t)(rows_total + 2) * 4));
    }
    ZDWB_TRY(rec_col.alloc(ctx, (size_t)(rec_cap + 1) * 4));
    ZDWB_TRY(rec_val.alloc(ctx, (size_t)(rec_cap + 1) * 8));
    if (delta) {
      ZDWB_TRY(chg_start.alloc(ctx, (size_t)(rec_cap + 1) * 4));
      ZDWB_TRY(chg_len.alloc(ctx, (size_t)(rec_cap + 1) * 4));
    }
    uint32_t cap_log2 = (uint32_t)std::max<long long>(10, std::min<long long>(ctx->ht_initial_log2, 31));
    while (cap_log2 < 31 && (1ull << cap_log2) < ctx->last_unique * 4) ++cap_log2;  // blocks of one file look alike
    if (!delta) {
      // a block cannot hold more distinct non-empty strings than non-empty fields
      uint32_t need = 10;
      while (need < 31 && (1ull << need) < ne_total * 2) ++need;
      if (cap_log2 > need) cap_log2 = need;
    }
    const uint32_t p1_tiles = (uint32_t)(((uint64_t)(-lo) + limit + tile_bytes - 1) / tile_bytes);
    bool bailed = false;
    for (;;) {
      const uint64_t cap = 1ull << cap_log2;
      ZDWB_TRY(slots.alloc(ctx, cap * 8));
      ZDWB_CUDA_TRY(ctx, cudaMemsetAsync(slots.p, 0, cap * 8, st));
      ht.slots = slots.as<unsigned long long>();
      ht.mask = (uint32_t)(cap - 1);
      ZDWB_TRY(launch(ctx, "k_init_minmax", k_init_minmax, (ncols + 255) / 256, 256, 0, colmin.as<unsigned long long>(),
                      colmax.as<unsigned long long>(), colset.as<uint32_t>(), ncols));
      P1Args A;
      A.buf = buf;
      A.n = n;
      A.lo = lo;
      A.limit = (int64_t)limit;
      A.ntiles = p1_tiles;
      A.ncols = ncols;
      A.pre = agg.as<TileAgg>();
      A.types = types_d.as<uint8_t>();
      A.trim = opts->trim_trailing_spaces;
      A.ht = ht;
      A.colset = colset.as<uint32_t>();
      A.colmin = colmin.as<unsigned long long>();
      A.colmax = colmax.as<unsigned long long>();
      A.rec_col = rec_col.as<uint32_t>();
      A.rec_val = rec_val.as<unsigned long long>();
      A.row_rec = census_free ? slot_rec.as<uint32_t>() : row_rec.as<uint32_t>();
      A.meta = meta;
      if (delta) {
        D1Args D;
        D.P = A;
        D.ntiles = p1_tiles;
        D.tile_bytes = tile_bytes;
        D.nrows = census_free ? (uint32_t)nslots : nrows;
        D.rec_cap = (uint32_t)rec_cap;
        D.row_cnt = census_free ? slot_cnt.as<uint32_t>() : row_cnt.as<uint32_t>();
        D.chg_start = chg_start.as<uint32_t>();
        D.chg_len = chg_len.as<uint32_t>();
        D.slot_cap = slot_cap;
        D.tile_rows = tile_rows.as<uint32_t>();
        const uint32_t d1_ctas = (p1_tiles + D1_WARPS - 1) / D1_WARPS;
        if (census_free)
          ZDWB_TRY(launch(ctx, "k_pass1d", k_pass1d<true>, d1_ctas, D1_THREADS, 0, D));
        else
          ZDWB_TRY(launch(ctx, "k_pass1d", k_pass1d<false>, d1_ctas, D1_THREADS, 0, D));
        D1List L;
        L.start = chg_start.as<uint32_t>();
        L.len = chg_len.as<uint32_t>();
        L.col = rec_col.as<uint32_t>();
        ZDWB_TRY(launch(ctx, "k_pass1d_values", k_pass1d_values, ctx->sm_count * 4, ENC_THREADS, 0, A, L, (uint32_t)rec_cap));
        if (census_free) {  // global row numbers; their total comes back with pass 1's read-back
          ZDWB_TRY(exclusive_scan_u32(ctx, tile_rows.as<uint32_t>(), tile_base.as<uint32_t>(), p1_tiles, &meta->tot_rows));
          ZDWB_TRY(launch(ctx, "k_row_fixup", k_row_fixup, (unsigned)((nslots + 255) / 256), 256, 0, tile_rows.as<uint32_t>(),
                          tile_base.as<uint32_t>(), p1_tiles, slot_cap, slot_rec.as<uint32_t>(), slot_cnt.as<uint32_t>(),
                          row_rec.as<uint32_t>(), row_cnt.as<uint32_t>(), meta));
        }
      } else {
        ZDWB_TRY(launch(ctx, "k_pass1", k_pass1, (p1_tiles + ENC_WARPS - 1) / ENC_WARPS, ENC_THREADS, 0, A));
      }
      // writeLookupColumnStats (ConvertToZDW.cpp:417-483) needs nothing from the host: it runs before the read-back
      ZDWB_TRY(launch(ctx, "k_col_stats", k_col_stats, 1, ENC_THREADS, 0, types_d.as<uint8_t>(), ncols, colset.as<uint32_t>(),
                      colmin.as<unsigned long long>(), colmax.as<unsigned long long>(), csize.as<uint8_t>(),
                      cbase.as<unsigned long long>(), used_idx.as<int32_t>(), used_cols.as<uint32_t>(), meta));
      if (delta) {  // the rows' places in the row stream; their total (the exact output size) comes back with the read-back
        const unsigned ctas = (unsigned)std::min<uint64_t>((rows_cap + ENC_WARPS - 1) / ENC_WARPS, (uint64_t)ctx->sm_count * 16);
        ZDWB_TRY(launch(ctx, "k_p2d_rowlen", k_p2d_rowlen, ctas, ENC_THREADS, 0, rec_col.as<uint32_t>(), row_rec.as<uint32_t>(),
                        row_cnt.as<uint32_t>(), (uint32_t)rows_cap, census_free, csize.as<uint8_t>(), meta, row_off.as<uint64_t>()));
        ZDWB_TRY(exclusive_scan_u64(ctx, row_off.as<uint64_t>(), row_off.as<uint64_t>(), rows_cap,
                                    reinterpret_cast<uint64_t*>(&meta->rows_bytes)));
      }
      ZDWB_CUDA_TRY(ctx, cudaMemcpyAsync(hmeta, meta, sizeof(EncMeta), cudaMemcpyDeviceToHost, st));
      ZDWB_CUDA_TRY(ctx, cudaStreamSynchronize(st));
      if (hmeta->delta_bail) {
        bailed = true;
        break;
      }
      if (hmeta->slot_overflow) break;
      if (hmeta->bad_row < (census_free ? hmeta->tot_rows : nrows)) break;
      const bool ht_full = hmeta->ht_overflow || hmeta->n_unique * 2 > cap;
      const bool rec_full = hmeta->rec_overflow != 0;
      if (!ht_full && !rec_full) break;
      if (ht_full) {
        if (cap_log2 >= 31) {
          ctx->err = "encode: dictionary hash set exceeds 2^31 slots";
          return ZDWB_ERR_UNSUPPORTED;
        }
        cap_log2 = std::min<uint32_t>(31, cap_log2 + 3);
      }
      if (rec_full) {
        rec_cap = std::min<uint64_t>(std::max<uint64_t>(rec_cap * 4, (uint64_t)hmeta->rec_count + 64), limit + 64);
        ZDWB_TRY(rec_col.alloc(ctx, (size_t)(rec_cap + 1) * 4));
        ZDWB_TRY(rec_val.alloc(ctx, (size_t)(rec_cap + 1) * 8));
        ZDWB_TRY(chg_start.alloc(ctx, (size_t)(rec_cap + 1) * 4));
        ZDWB_TRY(chg_len.alloc(ctx, (size_t)(rec_cap + 1) * 4));
      }
      // reset the counters pass 1 accumulates
      EncMeta z = *hmeta;
      z.ht_overflow = 0;
      z.rec_overflow = 0;
      z.rec_count = 0;
      z.n_unique = 0;
      z.dict_str_bytes = 0;
      z.max_str_len = 0;
      z.max_line = 0;
      *hmeta = z;
      ZDWB_CUDA_TRY(ctx, cudaMemcpyAsync(meta, hmeta, sizeof(EncMeta), cudaMemcpyHostToDevice, st));
      ZDWB_CUDA_TRY(ctx, cudaStreamSynchronize(st));
    }
    if (census_free) {
      int next = 0;
      if (bailed || hmeta->slot_overflow) {
        // A tile holds more rows than its slots, or a warp gave up: no row starts within the delta path's row limit
        // in front of its tile (a long run of blank lines, say), or a row runs past the limit (possibly the dropped
        // tail).  The census decides this block - it bails only where the row-delta pass cannot take the block - and
        // the context's later blocks take the census too, so that such a file does not run pass 1 twice a block.
        census_free = false;
        ctx->census_fell_back = true;
      } else {
        ZDWB_TRY(settle(&next));
        if (next == 1) return ZDWB_OK;
        if (next == 0) break;
        delta = census_free = false;
      }
      ZDWB_TRY(reset_meta());
      continue;
    }
    if (!bailed) break;
    // a row with more non-empty fields (or bytes) than a warp's lists hold: the whole block takes the general path
    delta = census_free = false;
    ctx->delta_bailed = true;
    ZDWB_TRY(reset_meta());
  }
  if (hmeta->bad_row < nrows) {
    out->bad_row = hmeta->bad_row + 1;  // "Row %u had the problem": one past the last good row, ConvertToZDW.cpp:811
    ctx->err = "Row " + std::to_string(out->bad_row) + " had the problem";
    return ZDWB_ERR_WRONG_COLUMNS;
  }
  if (probe) {
    // ---- the record at which the reference's string heap opens its K-th block
    const uint32_t nrec = (uint32_t)ne_total;
    probe->found = false;
    if (nrec) {
      DevBuf first_ord, new_len, pre, cut_d;
      const size_t cap = (size_t)ht.mask + 1;
      ZDWB_TRY(first_ord.alloc(ctx, cap * 4));
      ZDWB_TRY(new_len.alloc(ctx, (size_t)nrec * 8));
      ZDWB_TRY(pre.alloc(ctx, (size_t)nrec * 8));
      ZDWB_TRY(cut_d.alloc(ctx, sizeof(HeapCut)));
      ZDWB_CUDA_TRY(ctx, cudaMemsetAsync(first_ord.p, 0xff, cap * 4, st));
      ZDWB_TRY(launch(ctx, "k_heap_first_ord", k_heap_first_ord, (nrec + 255) / 256, 256, 0, rec_col.as<uint32_t>(),
                      rec_val.as<unsigned long long>(), types_d.as<uint8_t>(), nrec, first_ord.as<uint32_t>()));
      ZDWB_TRY(launch(ctx, "k_heap_new_len", k_heap_new_len, (nrec + 255) / 256, 256, 0, rec_col.as<uint32_t>(),
                      rec_val.as<unsigned long long>(), types_d.as<uint8_t>(), nrec, first_ord.as<uint32_t>(), ht.slots,
                      new_len.as<uint64_t>()));
      ZDWB_TRY(exclusive_scan_u64(ctx, new_len.as<uint64_t>(), pre.as<uint64_t>(), nrec, nullptr));
      ZDWB_TRY(launch(ctx, "k_heap_cut", k_heap_cut, 1, 1, 0, pre.as<uint64_t>(), new_len.as<uint64_t>(), nrec, 0, probe->K,
                      row_rec.as<uint32_t>(), nrows, rec_col.as<uint32_t>(), cut_d.as<HeapCut>()));
      HeapCut* hc = reinterpret_cast<HeapCut*>(reinterpret_cast<uint8_t*>(ctx->meta_host) + 2048);
      ZDWB_CUDA_TRY(ctx, cudaMemcpyAsync(hc, cut_d.p, sizeof(HeapCut), cudaMemcpyDeviceToHost, st));
      ZDWB_CUDA_TRY(ctx, cudaStreamSynchronize(st));
      probe->found = hc->found != 0;
      probe->row = hc->row;
      probe->col = hc->col;
      probe->allocs = hc->allocs;
    }
    return ZDWB_OK;
  }
  const uint64_t n_unique = hmeta->n_unique;
  ctx->last_unique = n_unique;
  if (delta) ctx->last_records = hmeta->rec_count;
  const uint64_t dict_total = hmeta->dict_str_bytes + 1;
  if (dict_total >= 0xffffffffull) {
    ctx->err = "encode: block dictionary would reach 4 GiB (Dictionary::size is 32-bit, dictionary.h:62); use smaller blocks";
    return ZDWB_ERR_UNSUPPORTED;
  }
  // the unterminated tail fills the row buffer the same way before being dropped (getnextrow.cpp:57-69)
  uint32_t max_line = hmeta->max_line;
  if (tail_bytes >= 2) max_line = std::max(max_line, tail_bytes + 1);
  max_line = std::max(max_line, spill_row_len);
  const uint32_t longest_field = longest_line_field(opts->prev_longest_line, max_line);

  // ---- column statistics: k_col_stats ran right behind pass 1, its results came back with pass 1's (one round trip)
  const uint32_t U = hmeta->n_used, nflag = hmeta->nflag;
  const uint64_t rows_base = hmeta->rows_base;

  // ---- dictionary order: compact the hash set, sort, offsets of the sorted entries, offset per slot
  DevBuf slot_off, ustart, ulen, uslot, order, offs;
  ZDWB_TRY(slot_off.alloc(ctx, ((size_t)ht.mask + 1) * 4));
  const uint32_t nu = (uint32_t)n_unique;
  if (nu) {
    ZDWB_TRY(ustart.alloc(ctx, (size_t)nu * 4));
    ZDWB_TRY(ulen.alloc(ctx, (size_t)nu * 4));
    ZDWB_TRY(uslot.alloc(ctx, (size_t)nu * 4));
    ZDWB_TRY(order.alloc(ctx, (size_t)nu * 4));
    ZDWB_TRY(offs.alloc(ctx, (size_t)nu * 4));
    const uint32_t cap = ht.mask + 1;
    ZDWB_TRY(launch(ctx, "k_ht_compact", k_ht_compact, (cap + ENC_THREADS - 1) / ENC_THREADS, ENC_THREADS, 0, ht.slots, cap,
                    ustart.as<uint32_t>(), ulen.as<uint32_t>(), uslot.as<uint32_t>(), meta));
    ZDWB_TRY(sort_strings(ctx, buf, ustart.as<uint32_t>(), ulen.as<uint32_t>(), nu, hmeta->max_str_len, order.as<uint32_t>()));
    ZDWB_TRY(launch(ctx, "k_sorted_lens", k_sorted_lens, (nu + 255) / 256, 256, 0, order.as<uint32_t>(), ulen.as<uint32_t>(), nu,
                    offs.as<uint32_t>()));
    ZDWB_TRY(exclusive_scan_u32(ctx, offs.as<uint32_t>(), offs.as<uint32_t>(), nu, nullptr));
    ZDWB_TRY(launch(ctx, "k_dict_slots", k_dict_slots, (nu + 255) / 256, 256, 0, order.as<uint32_t>(), uslot.as<uint32_t>(),
                    offs.as<uint32_t>(), nu, slot_off.as<uint32_t>()));
  }

  // ---- pass 2.  Row-delta: the row offsets are known already (k_p2d_rowlen), the rows are written into the output
  // below.  General: into the staging buffer, packed once every tile's length is known.
  uint64_t rows_bytes = delta ? hmeta->rows_bytes : 0;
  DevBuf staging, tile_bytes, tile_off, rows_total_d, colinfo;
  uint32_t tiles2 = 0;
  uint64_t tile_cap = 0;
  if (U > 0) {
    ZDWB_TRY(colinfo.alloc(ctx, (size_t)ncols * sizeof(ColInfo)));
    ZDWB_TRY(launch(ctx, "k_col_info", k_col_info, (ncols + 255) / 256, 256, 0, types_d.as<uint8_t>(), used_idx.as<int32_t>(),
                    cbase.as<unsigned long long>(), ncols, colinfo.as<ColInfo>()));
  }
  if (U > 0 && !delta) {
    // rows per CTA: bounded by the shared-memory value matrix ((R+1) * U * 8 bytes) and a record-count target
    if ((uint64_t)U * 8 * 2 + 1024 > 180 * 1024) {
      ctx->err = "encode: more than 11400 used columns in one block are not supported";
      return ZDWB_ERR_UNSUPPORTED;
    }
    const uint64_t smem_budget = 64 * 1024;
    const uint64_t by_smem = std::max<uint64_t>(2, smem_budget / ((uint64_t)U * 8));
    const uint64_t rec_per_row = std::max<uint64_t>(1, ne_total / std::max<uint64_t>(rows_total, 1));
    uint32_t rpc2 = (uint32_t)std::min<uint64_t>(std::max<uint64_t>(1, 4096 / rec_per_row), 1024);
    rpc2 = (uint32_t)std::min<uint64_t>(rpc2, by_smem - 1);
    if (ctx->enc_p2_rows > 0) rpc2 = (uint32_t)std::min<uint64_t>((uint64_t)ctx->enc_p2_rows, by_smem - 1);
    tiles2 = (nrows + rpc2 - 1) / rpc2;
    tile_cap = (((uint64_t)rpc2 * hmeta->max_row_bytes) + 15) & ~15ull;
    ZDWB_TRY(staging.alloc(ctx, (size_t)tiles2 * tile_cap + 64));
    ZDWB_TRY(tile_bytes.alloc(ctx, (size_t)tiles2 * 8));
    ZDWB_TRY(tile_off.alloc(ctx, (size_t)tiles2 * 8));
    ZDWB_TRY(rows_total_d.alloc(ctx, 8));
    const size_t smem = (size_t)(rpc2 + 1) * U * 8 + (size_t)(rpc2 + 1) * 4 + (size_t)(rpc2 + 2) * 4 + U + 16;
    ZDWB_CUDA_TRY(ctx, cudaFuncSetAttribute(k_pass2, cudaFuncAttributeMaxDynamicSharedMemorySize, 190 * 1024));
    ZDWB_TRY(launch(ctx, "k_pass2", k_pass2, tiles2, ENC_THREADS, smem, rec_col.as<uint32_t>(), rec_val.as<unsigned long long>(),
                    row_rec.as<uint32_t>(), nrows, rpc2, colinfo.as<ColInfo>(), slot_off.as<uint32_t>(), used_cols.as<uint32_t>(),
                    csize.as<uint8_t>(), U, nflag, tile_cap, staging.as<uint8_t>(), tile_bytes.as<uint64_t>()));
    ZDWB_TRY(exclusive_scan_u64(ctx, tile_bytes.as<uint64_t>(), tile_off.as<uint64_t>(), tiles2, rows_total_d.as<uint64_t>()));
    ZDWB_CUDA_TRY(ctx, cudaMemcpyAsync(reinterpret_cast<uint8_t*>(ctx->meta_host) + 1024, rows_total_d.p, 8, cudaMemcpyDeviceToHost, st));
    ZDWB_CUDA_TRY(ctx, cudaStreamSynchronize(st));
    memcpy(&rows_bytes, reinterpret_cast<uint8_t*>(ctx->meta_host) + 1024, 8);
  }

  // ---- output buffer of the exact size: header + dictionary + column stats, then the packed rows
  ctx->out_dev = nullptr;
  {
    DevBuf ob;
    ZDWB_TRY(ob.alloc(ctx, rows_base + rows_bytes + 64));
    ctx->out_dev = ob.detach();
  }
  uint8_t* outp = static_cast<uint8_t*>(ctx->out_dev);
  ZDWB_TRY(launch(ctx, "k_block_header", k_block_header, std::max(1u, std::min((ncols + 255) / 256, 64u)), 256, 0, outp, meta, nrows,
                  longest_field, is_last ? 1u : 0u, ncols, csize.as<uint8_t>(), cbase.as<unsigned long long>(), used_cols.as<uint32_t>()));
  if (nu) {
    const uint64_t threads = (uint64_t)nu * 8;
    ZDWB_TRY(launch(ctx, "k_dict_emit", k_dict_emit, (unsigned)((threads + 255) / 256), 256, 0, buf, order.as<uint32_t>(),
                    ustart.as<uint32_t>(), ulen.as<uint32_t>(), offs.as<uint32_t>(), nu, outp + hmeta->dict_base));
  }
  if (tiles2)
    ZDWB_TRY(launch(ctx, "k_gather_tiles", k_gather_tiles, tiles2, ENC_THREADS, 0, staging.as<uint8_t>(), tile_cap,
                    tile_off.as<uint64_t>(), tile_bytes.as<uint64_t>(), outp + rows_base));
  if (delta && rows_bytes) {
    const unsigned ctas = (unsigned)std::min<uint64_t>((nrows + ENC_WARPS - 1) / ENC_WARPS, (uint64_t)ctx->sm_count * 16);
    ZDWB_TRY(launch(ctx, "k_p2d_emit", k_p2d_emit, ctas, ENC_THREADS, 0, rec_col.as<uint32_t>(), rec_val.as<unsigned long long>(),
                    row_rec.as<uint32_t>(), row_cnt.as<uint32_t>(), row_off.as<uint64_t>(), nrows, nflag, colinfo.as<ColInfo>(),
                    csize.as<uint8_t>(), slot_off.as<uint32_t>(), outp + rows_base));
  }

  const size_t total_len = (size_t)(rows_base + rows_bytes);
  out->len = total_len;
  out->longest_line = longest_field;
  out->ncols_used = U;
  out->dict_entries = n_unique;
  out->dict_bytes = dict_total;
  out->dict_index_size = bytes_needed(dict_total);
  if (opts->output_on_device) {
    ZDWB_CUDA_TRY(ctx, cudaStreamSynchronize(st));
    out->bytes = outp;
  } else {
    if (ctx->out_host_cap < total_len) {
      out_host_release(ctx);
      size_t cap = std::max<size_t>(total_len + total_len / 4, 1 << 20);  // headroom: blocks of a file vary a little
      ZDWB_CUDA_TRY(ctx, cudaHostAlloc(&ctx->out_host, cap, cudaHostAllocDefault));
      ctx->out_host_pinned = true;
      ctx->out_host_cap = cap;
    }
    ZDWB_CUDA_TRY(ctx, cudaMemcpyAsync(ctx->out_host, outp, total_len, cudaMemcpyDeviceToHost, st));
    ZDWB_CUDA_TRY(ctx, cudaStreamSynchronize(st));
    out->bytes = static_cast<const uint8_t*>(ctx->out_host);
  }
  return ZDWB_OK;
}

}  // namespace zdwb
