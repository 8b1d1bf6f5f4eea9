// common.cuh -- shared device/host helpers for libzdw_b200 (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/zdw_b200.h"

namespace zdwb {

// ---------------------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------------------
struct Ctx {
  int device = 0;
  cudaStream_t own_stream = nullptr;
  cudaStream_t stream = nullptr;
  // device arena (arena_alloc / arena_release / arena_reset below): the scratch and the outputs of a call
  struct Chunk {
    uint8_t* p;
    size_t cap, used;
  };
  std::vector<Chunk> chunks;
  size_t arena_cur = 0;  // chunk allocations currently come from
  std::string err;
  unsigned long long launches = 0;
  int sm_count = 148;
  // tuning knobs
  long long small_sort_max = 65536;  // dictionaries up to this many entries are ranked by tile sort + binary search
  long long sort_radix_items = 0;    // records per thread in the radix passes: 4 or 16 (0 = by the number of records)
  long long ht_initial_log2 = 20;    // first-try size of the string hash set (grown x8 on overflow)
  long long dec_group_lanes = 0;     // lanes per strip in the row kernels: 8, 16, 32 (0 = by schema width)
  long long dec_strip_rows = 0;      // rows per strip of the row kernels (0 = automatic)
  long long copy_gate = 1;           // large H2D / D2H copies of different contexts take turns (0 = off)
  long long dec_delta = 1;           // wide schemas: rows are assembled from the row before (k_dec_write_delta)
  long long dec_tile_bytes = 8192;   // row-stream bytes per CTA in the decoder's row-boundary discovery
  unsigned long long last_out_per_row = 0;  // decoded bytes per row of the previous block (sizes the next output)
  unsigned long long last_unique = 0;  // dictionary size of the previous block (seeds the next hash set)
  long long enc_delta = -1;            // pass 1 variant: 1 = row-delta, 0 = general, -1 = by row width (encode.cu)
  long long enc_p2_rows = 0;           // rows per pass-2 tile (0 = automatic)
  long long enc_dtile = 0;             // bytes per row-delta tile (0 = automatic; a power of two >= 2048)
  long long enc_census = -1;           // row-delta row census: 1 = always, 0 = skipped for every uncut block, -1 = automatic
  bool delta_bailed = false;           // a block of this context did not fit the row-delta pass: stop trying
  bool census_fell_back = false;       // a census-free pass 1 of this context handed its block to the census
  unsigned long long last_row_bytes = 0;  // mean row length of the previous block
  unsigned long long last_records = 0;    // records the previous block's row-delta pass 1 produced (sizes the next arrays)
  // outputs owned by the context (valid until the next call)
  void* out_dev = nullptr;     // device output buffer
  void* out_dev2 = nullptr;    // second device output (row offsets)
  void* out_host = nullptr;    // host output: pinned, or plain malloc'd memory for a one-off result (out_host_pinned)
  size_t out_host_cap = 0;
  bool out_host_pinned = true;
  unsigned long long decode_calls = 0;  // host-output decode calls served so far
  void* out_host2 = nullptr;
  size_t out_host2_cap = 0;
  std::vector<unsigned long long> flag_counts;  // -s statistics of the last decoded block
  // pinned staging ring (ring_h2d / ring_d2h below): pageable caller memory and file descriptors reach the device through
  // it in chunks, the copy of one chunk under the host's work on the next
  static constexpr int RING_SLOTS = 3;
  static constexpr size_t RING_CHUNK = (size_t)8 << 20;
  void* ring_buf[RING_SLOTS] = {nullptr, nullptr, nullptr};
  cudaEvent_t ring_ev[RING_SLOTS] = {nullptr, nullptr, nullptr};
  bool ring_busy[RING_SLOTS] = {false, false, false};
  void* fd_dev = nullptr;      // device buffer of zdwb_fd_to_device (own allocation: it outlives the arena resets of the calls)
  size_t fd_dev_cap = 0;
  // pinned arena for the small tables of a call (schema, widths, output template): copies from pageable memory go
  // through the driver's own staging and serialise with other driver work; from here they are plain async copies
  void* stage_host = nullptr;
  size_t stage_cap = 0, stage_used = 0;
  // small pinned scratch for device->host readbacks of metadata
  void* meta_host = nullptr;
  // optional per-kernel timing (CUDA events on the launching stream), for the roofline report
  bool timing = false;
  struct Timed {
    const char* name;
    cudaEvent_t e0, e1;
  };
  std::vector<Timed> timed;
};

#define ZDWB_CUDA_TRY(ctx, expr)                                                                   \
  do {                                                                                             \
    cudaError_t _e = (expr);                                                                       \
    if (_e != cudaSuccess) {                                                                       \
      char _b[512];                                                                                \
      snprintf(_b, sizeof(_b), "%s:%d: %s failed: %s", __FILE__, __LINE__, #expr,                  \
               cudaGetErrorString(_e));                                                            \
      (ctx)->err = _b;                                                                             \
      (void)cudaGetLastError();                                                                    \
      return (_e == cudaErrorMemoryAllocation) ? ZDWB_ERR_OOM : ZDWB_ERR_CUDA;                      \
    }                                                                                              \
  } while (0)

#define ZDWB_TRY(expr)                    \
  do {                                    \
    int _rc = (expr);                     \
    if (_rc != ZDWB_OK) return _rc;       \
  } while (0)

#ifdef __CUDACC__
// Launches kernel k on the context's stream: bracketed by events when Ctx::timing is on, counted in Ctx::launches, and
// checked for launch errors, which name the kernel in Ctx::err.
template <class... P, class... A>
int launch(Ctx* c, const char* name, void (*k)(P...), dim3 grid, dim3 block, size_t smem, A... args) {
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  if (c->timing) {
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    cudaEventRecord(e0, c->stream);
  }
  k<<<grid, block, smem, c->stream>>>(args...);
  if (e0) {
    cudaEventRecord(e1, c->stream);
    c->timed.push_back(Ctx::Timed{name, e0, e1});
  }
  ++c->launches;
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    c->err = std::string("launch of ") + name + " failed: " + cudaGetErrorString(e);
    return e == cudaErrorMemoryAllocation ? ZDWB_ERR_OOM : ZDWB_ERR_CUDA;
  }
  return ZDWB_OK;
}
#endif

// Device memory of a call comes from a per-context stack arena: a few big cudaMalloc'd chunks that every call re-uses
// from the bottom, so a call in steady state makes no driver-level memory-management call at all (those serialise with
// other driver work such as NVML queries, and cost host time per block).  Allocation bumps the top of the current
// chunk; scoped buffers die in reverse order of construction, so releasing the top one pops it and the space is
// re-used within the call (everything runs on the context's one stream, so re-use is ordered).  When the current chunk
// is full the arena moves on to the next one that is empty and large enough, or adds one; chunks are kept for the
// life of the context, so the second call of a kind already finds what the first one needed.
inline void* arena_alloc(Ctx* c, size_t n) {
  n = (n + 255) & ~(size_t)255;
  for (;;) {
    if (c->arena_cur < c->chunks.size()) {
      Ctx::Chunk& k = c->chunks[c->arena_cur];
      if (k.used + n <= k.cap) {
        void* r = k.p + k.used;
        k.used += n;
        return r;
      }
      // later chunks are empty (stack discipline): take the first one that is large enough
      size_t j = c->arena_cur + 1;
      while (j < c->chunks.size() && c->chunks[j].cap < n) ++j;
      if (j < c->chunks.size()) {
        if (j != c->arena_cur + 1) std::swap(c->chunks[j], c->chunks[c->arena_cur + 1]);
        ++c->arena_cur;
        continue;
      }
    }
    size_t total = 0;
    for (const Ctx::Chunk& k : c->chunks) total += k.cap;
    size_t cap = std::max<size_t>(n, std::max<size_t>((size_t)64 << 20, total / 2));
    void* p = nullptr;
    if (cudaMalloc(&p, cap) != cudaSuccess) {
      (void)cudaGetLastError();
      if (cap == n || cudaMalloc(&p, n) != cudaSuccess) {
        (void)cudaGetLastError();
        return nullptr;
      }
      cap = n;
    }
    c->chunks.push_back(Ctx::Chunk{static_cast<uint8_t*>(p), cap, 0});
    if (c->chunks.size() > 1 && c->arena_cur + 1 != c->chunks.size() - 1)
      std::swap(c->chunks.back(), c->chunks[c->arena_cur + 1]);
    c->arena_cur = c->chunks.size() == 1 ? 0 : c->arena_cur + 1;
  }
}
inline void arena_release(Ctx* c, void* p, size_t n) {
  n = (n + 255) & ~(size_t)255;
  if (c->arena_cur >= c->chunks.size()) return;
  Ctx::Chunk& k = c->chunks[c->arena_cur];
  if (static_cast<uint8_t*>(p) + n == k.p + k.used) {  // the top allocation: pop it
    k.used -= n;
    if (k.used == 0 && c->arena_cur > 0) --c->arena_cur;
  }  // anything else stays until the next reset
}
// Start of a call: everything handed out before (including the previous call's outputs) is gone.
inline int arena_reset(Ctx* c) {
  for (Ctx::Chunk& k : c->chunks) k.used = 0;
  c->arena_cur = 0;
  return ZDWB_OK;
}
inline void arena_destroy(Ctx* c) {
  for (const Ctx::Chunk& k : c->chunks) cudaFree(k.p);
  c->chunks.clear();
}

// Scoped device allocation from the context's arena.
struct DevBuf {
  Ctx* ctx = nullptr;
  void* p = nullptr;
  size_t bytes = 0;
  DevBuf() {}
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { release(); }
  int alloc(Ctx* c, size_t n) {
    release();
    ctx = c;
    bytes = n ? n : 16;
    p = arena_alloc(c, bytes);
    if (!p) {
      char b[256];
      snprintf(b, sizeof(b), "device allocation of %zu bytes failed", bytes);
      c->err = b;
      return ZDWB_ERR_OOM;
    }
    return ZDWB_OK;
  }
  void release() {
    if (p) {
      arena_release(ctx, p, bytes);
      p = nullptr;
    }
  }
  void* detach() {  // the buffer outlives this object: it stays valid until the next call on the context
    void* q = p;
    p = nullptr;
    return q;
  }
  template <typename T>
  T* as() const {
    return reinterpret_cast<T*>(p);
  }
};

// Large host<->device copies of one direction take turns, process-wide per device.  Contexts that work on different
// blocks at the same time otherwise fall into step: their copies share the link, finish together, then all of them
// run kernels while the link idles (measured with three contexts: 11.3 ms per 504 MB block instead of the 9.1 ms the
// link needs).  One copy at a time finishes earlier, its kernels then run under the next context's copy.
inline std::mutex& copy_gate(int device, int dir) {
  static std::mutex gates[2][64];
  return gates[dir & 1][(unsigned)device & 63u];
}
constexpr size_t COPY_GATE_MIN = (size_t)8 << 20;  // smaller copies are not worth a turn

// host output buffer of the context (see Ctx::out_host)
inline void out_host_release(Ctx* c) {
  if (c->out_host) {
    if (c->out_host_pinned) cudaFreeHost(c->out_host);
    else free(c->out_host);
  }
  c->out_host = nullptr;
  c->out_host_cap = 0;
}

// Pinned arena of the context: stage_reset() at the start of a call (the stream is idle then), stage_take() hands out
// 16-byte aligned pieces that stay valid until the next reset.
inline int stage_reset(Ctx* c) {
  if (c->stage_used) {
    cudaError_t e = cudaStreamSynchronize(c->stream);  // copies of an earlier call that ended early
    if (e != cudaSuccess) {
      c->err = std::string("cudaStreamSynchronize failed: ") + cudaGetErrorString(e);
      (void)cudaGetLastError();
      return ZDWB_ERR_CUDA;
    }
  }
  c->stage_used = 0;
  return ZDWB_OK;
}
// start of an encode / decode call
inline int call_begin(Ctx* c) {
  int rc = stage_reset(c);
  if (rc != ZDWB_OK) return rc;
  return arena_reset(c);
}
inline void* stage_take(Ctx* c, size_t n) {
  const size_t need = (n + 15) & ~(size_t)15;
  if (c->stage_used + need > c->stage_cap) {
    // grow: pieces already handed out must stay valid, so the old arena is only released once the stream is idle
    size_t cap = c->stage_cap ? c->stage_cap * 2 : (size_t)1 << 20;
    while (cap < need) cap *= 2;
    void* p = nullptr;
    if (cudaHostAlloc(&p, cap, cudaHostAllocDefault) != cudaSuccess) {
      (void)cudaGetLastError();
      return nullptr;
    }
    if (c->stage_host) {
      cudaStreamSynchronize(c->stream);
      cudaFreeHost(c->stage_host);
    }
    c->stage_host = p;
    c->stage_cap = cap;
    c->stage_used = 0;
  }
  void* r = static_cast<uint8_t*>(c->stage_host) + c->stage_used;
  c->stage_used += need;
  return r;
}

// ---- pinned staging ring --------------------------------------------------------------------------------------
// A copy straight from / to pageable memory goes through the driver's own staging at 2-3 GB/s (measured: 0.42 s for a
// 1 GiB window, 0.5 s for 1 GiB of decoded rows) and a window-sized pinned buffer costs 0.45 s per GiB to allocate; three
// 8 MiB pinned chunks cost nothing and keep the link busy while the host fills or drains the chunk next to it.
inline int ring_init(Ctx* c) {
  for (int k = 0; k < Ctx::RING_SLOTS; ++k) {
    if (!c->ring_buf[k]) {
      if (cudaHostAlloc(&c->ring_buf[k], Ctx::RING_CHUNK, cudaHostAllocDefault) != cudaSuccess) {
        (void)cudaGetLastError();
        c->ring_buf[k] = nullptr;
        c->err = "pinned staging ring allocation failed";
        return ZDWB_ERR_OOM;
      }
    }
    if (!c->ring_ev[k] && cudaEventCreateWithFlags(&c->ring_ev[k], cudaEventDisableTiming) != cudaSuccess) {
      (void)cudaGetLastError();
      c->ring_ev[k] = nullptr;
      c->err = "cudaEventCreate failed";
      return ZDWB_ERR_CUDA;
    }
  }
  return ZDWB_OK;
}
inline void ring_destroy(Ctx* c) {
  for (int k = 0; k < Ctx::RING_SLOTS; ++k) {
    if (c->ring_ev[k]) cudaEventDestroy(c->ring_ev[k]);
    if (c->ring_buf[k]) cudaFreeHost(c->ring_buf[k]);
    c->ring_ev[k] = nullptr;
    c->ring_buf[k] = nullptr;
    c->ring_busy[k] = false;
  }
}
// host -> device: fill(dst, offset, n) puts bytes [offset, offset + n) of the source into dst (false = failed).  The
// copies are queued on the context's stream; nothing waits for the last ones (the kernels behind them do).
template <class Fill>
inline int ring_h2d(Ctx* c, void* dev, size_t len, Fill fill) {
  ZDWB_TRY(ring_init(c));
  size_t i = 0;
  for (size_t off = 0; off < len; off += Ctx::RING_CHUNK, ++i) {
    const int k = (int)(i % Ctx::RING_SLOTS);
    if (c->ring_busy[k]) ZDWB_CUDA_TRY(c, cudaEventSynchronize(c->ring_ev[k]));
    c->ring_busy[k] = false;
    const size_t n = std::min(Ctx::RING_CHUNK, len - off);
    if (!fill(c->ring_buf[k], off, n)) {
      if (c->err.empty()) c->err = "reading the input failed";
      return ZDWB_ERR_BAD_ARG;
    }
    ZDWB_CUDA_TRY(c, cudaMemcpyAsync(static_cast<uint8_t*>(dev) + off, c->ring_buf[k], n, cudaMemcpyHostToDevice, c->stream));
    ZDWB_CUDA_TRY(c, cudaEventRecord(c->ring_ev[k], c->stream));
    c->ring_busy[k] = true;
  }
  return ZDWB_OK;
}
// device -> host: drain(src, offset, n) takes bytes [offset, offset + n) of the device range (false = failed).  Two
// copies are in flight while a chunk is drained; returns when everything has been drained.
template <class Drain>
inline int ring_d2h(Ctx* c, const void* dev, size_t len, Drain drain) {
  ZDWB_TRY(ring_init(c));
  const size_t nch = (len + Ctx::RING_CHUNK - 1) / Ctx::RING_CHUNK;
  for (int k = 0; k < Ctx::RING_SLOTS; ++k) {
    if (c->ring_busy[k]) ZDWB_CUDA_TRY(c, cudaEventSynchronize(c->ring_ev[k]));
    c->ring_busy[k] = false;
  }
  for (size_t i = 0; i < nch + 2; ++i) {
    if (i < nch) {
      const int k = (int)(i % Ctx::RING_SLOTS);
      const size_t off = i * Ctx::RING_CHUNK, n = std::min(Ctx::RING_CHUNK, len - off);
      ZDWB_CUDA_TRY(c, cudaMemcpyAsync(c->ring_buf[k], static_cast<const uint8_t*>(dev) + off, n, cudaMemcpyDeviceToHost, c->stream));
      ZDWB_CUDA_TRY(c, cudaEventRecord(c->ring_ev[k], c->stream));
    }
    if (i >= 2) {
      const size_t j = i - 2;
      const int k = (int)(j % Ctx::RING_SLOTS);
      const size_t off = j * Ctx::RING_CHUNK, n = std::min(Ctx::RING_CHUNK, len - off);
      ZDWB_CUDA_TRY(c, cudaEventSynchronize(c->ring_ev[k]));
      if (!drain(static_cast<const uint8_t*>(c->ring_buf[k]), off, n)) {
        cudaStreamSynchronize(c->stream);  // (copies into the ring that are still under way)
        if (c->err.empty()) c->err = "writing the output failed";
        return ZDWB_ERR_BAD_ARG;
      }
    }
  }
  return ZDWB_OK;
}
// is p ordinary (unregistered, pageable) host memory?
inline bool is_pageable_host(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    (void)cudaGetLastError();
    return true;
  }
  return a.type == cudaMemoryTypeUnregistered;
}

// ---------------------------------------------------------------------------------------------
// column types
// ---------------------------------------------------------------------------------------------
// "dictionary" types: ConvertToZDW.cpp:345-352
__host__ __device__ __forceinline__ bool is_text_like(uint8_t t) {
  return t == ZDWB_DECIMAL || t == ZDWB_VARCHAR || t == ZDWB_TEXT || t == ZDWB_TINYTEXT ||
         t == ZDWB_MEDIUMTEXT || t == ZDWB_LONGTEXT || t == ZDWB_DATETIME || t == ZDWB_CHAR_2;
}
__host__ __device__ __forceinline__ bool is_int_type(uint8_t t) {
  return (t >= ZDWB_TINY && t <= ZDWB_LONGLONG) || (t >= ZDWB_TINY_SIGNED && t <= ZDWB_LONGLONG_SIGNED);
}
__host__ __device__ __forceinline__ bool is_signed_int_type(uint8_t t) {
  return t >= ZDWB_TINY_SIGNED && t <= ZDWB_LONGLONG_SIGNED;
}
__host__ __device__ __forceinline__ bool is_known_type(uint8_t t) {
  return is_text_like(t) || is_int_type(t) || t == ZDWB_CHAR;
}

// ---------------------------------------------------------------------------------------------
// numeric semantics shared by kernels and host-side unit tests
// ---------------------------------------------------------------------------------------------

// strtoull(f, NULL, 10) over a bounded field (ConvertToZDW.cpp:385,564; SURVEY App. B-5/B-24): skip
// isspace() bytes, optional sign, digits; overflow saturates to 2^64-1 regardless of sign; a '-'
// negates modulo 2^64.  Bytes past `len` read as NUL (the reference NUL-terminates every field).
__host__ __device__ __forceinline__ uint64_t parse_u64_field(const uint8_t* p, uint32_t len) {
  uint32_t i = 0;
  while (i < len) {
    uint8_t ch = p[i];
    if (ch == ' ' || (ch >= 9 && ch <= 13)) ++i;
    else break;
  }
  bool neg = false;
  if (i < len && (p[i] == '+' || p[i] == '-')) {
    neg = p[i] == '-';
    ++i;
  }
  uint64_t v = 0;
  bool ovf = false;
  while (i < len) {
    uint32_t d = (uint32_t)p[i] - (uint32_t)'0';
    if (d > 9) break;
    // v*10 + d > 2^64-1 ?
    if (v > 1844674407370955161ULL || (v == 1844674407370955161ULL && d > 5)) ovf = true;
    v = v * 10 + d;
    ++i;
  }
  if (ovf) return ~0ULL;
  return neg ? (0 - v) : v;
}

// CHAR column value: sign-extended first byte (+ second byte * 256).  `second_always` selects the
// pass-2 rule (ConvertToZDW.cpp:543-547: add f[1]*256 whenever f[0] != 0) over the pass-1 rule
// (:359-361: only when f[0] == '\\').  f[1] reads as NUL for a 1-byte field.
__host__ __device__ __forceinline__ uint64_t char_tuple(const uint8_t* p, uint32_t len, bool second_always) {
  if (len == 0) return 0;
  int64_t v = (int64_t)(int8_t)p[0];
  if (second_always || p[0] == '\\') {
    int32_t b1 = len > 1 ? (int32_t)(int8_t)p[1] : 0;
    v += (int64_t)(b1 * 256);
  }
  return (uint64_t)v;
}

// bytes needed to store v (1..8): ConvertToZDW.cpp:458-465, dictionary.cpp:62-73
__host__ __device__ __forceinline__ uint32_t bytes_needed(uint64_t v) {
  uint32_t k = 1;
  while (v >= 256) {
    ++k;
    v >>= 8;
  }
  return k;
}

// llutoa (UnconvertFromZDW.cpp:318-330): writes digits ending at `end` (exclusive), returns length.
__host__ __device__ __forceinline__ uint32_t fmt_u64(uint64_t v, uint8_t* end) {
  uint8_t* p = end;
  do {
    *--p = (uint8_t)('0' + (v % 10));
    v /= 10;
  } while (v);
  return (uint32_t)(end - p);
}

// lltoa (UnconvertFromZDW.cpp:333-356) including its INT64_MIN behaviour (SURVEY App. B-22): the
// negation overflows, every `value % 10` is then <= 0 and the digit byte is 0x30 + rem.
__host__ __device__ __forceinline__ uint32_t fmt_i64(int64_t sv, uint8_t* end) {
  uint8_t* p = end;
  bool minus = false;
  if (sv < 0) {
    minus = true;
    sv = (int64_t)(0 - (uint64_t)sv);
  }
  do {
    int64_t rem = sv % 10;
    sv /= 10;
    *--p = (uint8_t)(rem + 0x30);
  } while (sv != 0);
  if (minus) *--p = '-';
  return (uint32_t)(end - p);
}

// four decimal digits of x (< 10000) as ASCII, most significant digit in the lowest byte: two 2-digit fields are split
// into tens and ones side by side (x / 100 = x * 5243 >> 19 for x < 43699, y / 10 = y * 103 >> 10 for y < 179)
__host__ __device__ __forceinline__ uint32_t ascii4(uint32_t x) {
  const uint32_t hi = (x * 5243u) >> 19;
  const uint32_t p = hi | ((x - hi * 100u) << 16);
  const uint32_t tens = ((p * 103u) >> 10) & 0x000f000fu;
  const uint32_t ones = p - tens * 10u;
  return (tens | (ones << 8)) + 0x30303030u;
}

#ifdef __CUDA_ARCH__
#define ZDWB_FUNNEL_R(lo, hi, sh) __funnelshift_r((lo), (hi), (sh))
#else
#define ZDWB_FUNNEL_R(lo, hi, sh) ((uint32_t)((((uint64_t)(hi) << 32) | (uint64_t)(lo)) >> ((sh) & 31u)))
#endif

// Decimal text of `full` as llutoa / lltoa print it (UnconvertFromZDW.cpp:318-356), exactly len characters, left-aligned
// in w[0..4] (the first character is the lowest byte of w[0]); bytes past len are unspecified.  Straight-line: the 20
// zero-padded digits are produced four at a time and the leading zeros shifted out.  `neg` = the value prints with a
// minus sign (len counts it); INT64_MIN keeps the reference's digits 0x30 - d (SURVEY App. B-22).
__host__ __device__ __forceinline__ void render_int(unsigned long long full, bool neg, uint32_t len, uint32_t w[5]) {
  const unsigned long long mag = neg ? 0ull - full : full;
  uint32_t a, b, c;
  if (mag <= 0xffffffffull) {
    const uint32_t x = (uint32_t)mag;
    a = 0;
    b = x / 100000000u;
    c = x - b * 100000000u;
  } else {
    const unsigned long long q = mag / 100000000ull;
    c = (uint32_t)(mag - q * 100000000ull);
    const unsigned long long q2 = q / 100000000ull;
    b = (uint32_t)(q - q2 * 100000000ull);
    a = (uint32_t)q2;
  }
  const uint32_t bh = b / 10000u, ch = c / 10000u;
  uint32_t e0 = ascii4(a), e1 = ascii4(bh), e2 = ascii4(b - bh * 10000u), e3 = ascii4(ch), e4 = ascii4(c - ch * 10000u);
  if (neg && full == 0x8000000000000000ull) {  // every remainder is negative: digit byte = 0x30 - d
    e0 = 0x60606060u - e0;
    e1 = 0x60606060u - e1;
    e2 = 0x60606060u - e2;
    e3 = 0x60606060u - e3;
    e4 = 0x60606060u - e4;
  }
  const uint32_t nd = len - (neg ? 1u : 0u);  // digits
  const uint32_t s = 20u - nd, ws = s >> 2, bs = (s & 3u) * 8u;
  if (ws & 4u) e0 = e4;
  if (ws & 2u) {
    e0 = e2;
    e1 = e3;
    e2 = e4;
  }
  if (ws & 1u) {
    e0 = e1;
    e1 = e2;
    e2 = e3;
    e3 = e4;
  }
  uint32_t x0 = ZDWB_FUNNEL_R(e0, e1, bs), x1 = ZDWB_FUNNEL_R(e1, e2, bs), x2 = ZDWB_FUNNEL_R(e2, e3, bs),
           x3 = ZDWB_FUNNEL_R(e3, e4, bs), x4 = e4 >> bs;
  if (neg) {  // make room for the sign
    x4 = (x4 << 8) | (x3 >> 24);
    x3 = (x3 << 8) | (x2 >> 24);
    x2 = (x2 << 8) | (x1 >> 24);
    x1 = (x1 << 8) | (x0 >> 24);
    x0 = (x0 << 8) | (uint32_t)'-';
  }
  w[0] = x0;
  w[1] = x1;
  w[2] = x2;
  w[3] = x3;
  w[4] = x4;
}

// strtoull of a field of 1..20 bytes that consists of decimal digits only, from its masked words - the common case;
// everything else (whitespace, signs, junk, 21+ characters) takes parse_u64_field.  Twenty digits can exceed 2^64 - 1:
// strtoull then saturates (SURVEY App. B-5).  Returns false when the field is not all digits.
constexpr uint32_t NUM_FAST_MAX = 20;
__host__ __device__ __forceinline__ bool digits_value(const uint32_t x[5], uint32_t len, unsigned long long* out) {
  unsigned long long v = 0;
  bool ok = true, ovf = false;
#pragma unroll
  for (uint32_t k = 0; k < 5; ++k) {
    if (4u * k < len) {
      const uint32_t nd = len - 4u * k < 4u ? len - 4u * k : 4u;
      const uint32_t keep = nd >= 4u ? 0xffffffffu : ((1u << (8u * nd)) - 1u);
      const uint32_t w = (x[k] & keep) | (0x30303030u & ~keep);       // pad with '0'
      const uint32_t d = w - 0x30303030u;
      ok = ok && (((w + 0x46464646u) | d) & 0x80808080u) == 0u;        // every byte in '0'..'9'
      const uint32_t al = nd >= 4u ? d : (d << (8u * (4u - nd)));      // right-align: leading zero digits
      const uint32_t pairs = (al & 0x00ff00ffu) * 10u + ((al >> 8) & 0x00ff00ffu);
      const uint32_t v4 = (pairs & 0xffffu) * 100u + (pairs >> 16);
      const uint32_t scale = nd == 4u ? 10000u : nd == 3u ? 1000u : nd == 2u ? 100u : 10u;
      if (k == 4u && nd == 4u)  // the 17th..20th digit: v * 10^4 + v4 > 2^64 - 1 ?
        ovf = v > 1844674407370955ull || (v == 1844674407370955ull && v4 > 1615u);
      v = v * scale + v4;
    }
  }
  *out = ovf ? ~0ull : v;
  return ok;
}

// strtoull of a field of 1..20 bytes held in five masked little-endian words (bytes past `len` are zero): an optional
// sign in front of the digits ('-' negates modulo 2^64; with a sign at most 19 digits are left, which cannot overflow).
// Returns false for anything else - white space, junk, a lone sign - which takes the exact byte walk parse_u64_field.
__host__ __device__ __forceinline__ bool fast_number(const uint32_t x[5], uint32_t len, unsigned long long* out) {
  const uint32_t c0 = x[0] & 0xffu;
  const bool sign = c0 == (uint32_t)'-' || c0 == (uint32_t)'+';
  uint32_t y[5] = {x[0], x[1], x[2], x[3], x[4]};
  uint32_t dl = len;
  if (sign) {
    y[0] = ZDWB_FUNNEL_R(x[0], x[1], 8u);
    y[1] = ZDWB_FUNNEL_R(x[1], x[2], 8u);
    y[2] = ZDWB_FUNNEL_R(x[2], x[3], 8u);
    y[3] = ZDWB_FUNNEL_R(x[3], x[4], 8u);
    y[4] = x[4] >> 8;
    dl = len - 1u;
  }
  unsigned long long v;
  if (dl == 0u || !digits_value(y, dl, &v)) return false;
  *out = c0 == (uint32_t)'-' ? 0ull - v : v;
  return true;
}

// ---------------------------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------------------------
#ifdef __CUDACC__

__device__ __forceinline__ unsigned lane_id() { return threadIdx.x & 31; }
__device__ __forceinline__ unsigned lanemask_lt() {
  unsigned m;
  asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
  return m;
}

// streaming 16-byte load that does not allocate in L1 (each TSV byte is consumed once per pass)
__device__ __forceinline__ uint4 ldg_stream_u4(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}
// 16-byte load of bytes that are read again soon (the row-delta pass compares every row with the one before it).
// The no-allocate form above is treated as evict-first by L2 as well: with it 80 % of the TSV came from DRAM twice
// (ncu: 905 MB read for a 504 MB block), the second time with DRAM latency in front of the compares.
__device__ __forceinline__ uint4 ldg_keep_u4(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

__device__ __forceinline__ uint64_t ld_acquire_u64(const uint64_t* p) {
  uint64_t v;
  asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_u64(uint64_t* p, uint64_t v) {
  asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ uint64_t ld_relaxed_u64(const uint64_t* p) {
  uint64_t v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}

// ---- bulk asynchronous copies (TMA, 1-D) global -> shared with an mbarrier that counts the bytes that have landed.
// One lane arms the barrier with the byte count and issues the copy; every consumer waits for the barrier's phase.
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t arrivals) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(arrivals) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_load(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
    "{\n"
    ".reg .pred p;\n"
    "WAIT_LOOP:\n"
    "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
    "@p bra WAIT_DONE;\n"
    "bra WAIT_LOOP;\n"
    "WAIT_DONE:\n"
    "}\n" ::"r"(smem_u32(bar)),
    "r"(parity)
    : "memory");
}
// orders the generic-proxy accesses of this thread before later async-proxy (bulk copy) accesses to shared memory
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// decimal digits of x (llutoa's text length)
__device__ __forceinline__ uint32_t digits_u32(uint32_t x) {
  return x < 10u ? 1u : x < 100u ? 2u : x < 1000u ? 3u : x < 10000u ? 4u : x < 100000u ? 5u : x < 1000000u ? 6u
         : x < 10000000u ? 7u : x < 100000000u ? 8u : x < 1000000000u ? 9u : 10u;
}
__device__ __forceinline__ uint32_t digits_u64(unsigned long long v) {
  if (v <= 0xffffffffull) return digits_u32((uint32_t)v);
  if (v < 100000000000000ull) {  // < 10^14
    return v < 10000000000ull ? 10u : v < 100000000000ull ? 11u : v < 1000000000000ull ? 12u : v < 10000000000000ull ? 13u : 14u;
  }
  return v < 1000000000000000ull ? 15u : v < 10000000000000000ull ? 16u : v < 100000000000000000ull ? 17u
         : v < 1000000000000000000ull ? 18u : v < 10000000000000000000ull ? 19u : 20u;
}

// a string in device memory (merge.cu, match.cu)
struct Str {
  const uint8_t* p;
  unsigned long long len;
};

// bytes [off, off + 8) of s as a big-endian number, zero past len (the idea of sort.cu's prefix_key)
__device__ __forceinline__ unsigned long long key8(const uint8_t* s, unsigned long long len, unsigned long long off) {
  unsigned long long k = 0;
#pragma unroll
  for (uint32_t i = 0; i < 8; ++i) k = (k << 8) | (off + i < len ? (unsigned long long)__ldg(s + off + i) : 0ull);
  return k;
}

// bytewise order (memcmp over the shorter, then the length); the keys hold bytes 0..15
__device__ __forceinline__ int str_cmp(const ulonglong2& ka, const Str& a, const ulonglong2& kb, const Str& b) {
  if (ka.x != kb.x) return ka.x < kb.x ? -1 : 1;
  if (ka.y != kb.y) return ka.y < kb.y ? -1 : 1;
  // 8 bytes at a time past the keys: a word that straddles the shorter length compares its zero padding with the
  // longer string's bytes, which orders the pair as the length compare below would, or finds them equal
  const unsigned long long m = a.len < b.len ? a.len : b.len;
  for (unsigned long long i = 16; i < m; i += 8) {
    const unsigned long long x = key8(a.p, a.len, i), y = key8(b.p, b.len, i);
    if (x != y) return x < y ? -1 : 1;
  }
  return a.len < b.len ? -1 : a.len > b.len ? 1 : 0;
}

// per-byte equality mask of a 32-bit word against a replicated byte: bit 7 of each byte lane set
__device__ __forceinline__ uint32_t bytes_eq(uint32_t w, uint32_t rep) {
  uint32_t x = w ^ rep;
  // zero-byte detect, exact variant (no false positives across byte lanes)
  return ~(((x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | x | 0x7F7F7F7Fu);
}
// gather the four bit-7 flags of a word into the low 4 bits: (m >> 7) has bits 0/8/16/24; the multiplier
// 2^21 + 2^14 + 2^7 + 1 moves them to bits 21..24 and no two partial products share a bit (no carries)
__device__ __forceinline__ uint32_t movemask4(uint32_t m) { return (((m >> 7) * 0x00204081u) >> 21) & 0xFu; }
// 16-bit mask of bytes equal to `ch` within a 16-byte chunk
__device__ __forceinline__ uint32_t chunk_mask(const uint4& v, uint8_t ch) {
  const uint32_t rep = 0x01010101u * ch;
  return movemask4(bytes_eq(v.x, rep)) | (movemask4(bytes_eq(v.y, rep)) << 4) |
         (movemask4(bytes_eq(v.z, rep)) << 8) | (movemask4(bytes_eq(v.w, rep)) << 12);
}
// does the 16-byte chunk hold any byte equal to `ch`?  ((x - 0x01..) & ~x & 0x80..) is exact as an any-test
__device__ __forceinline__ bool chunk_has(const uint4& v, uint8_t ch) {
  const uint32_t rep = 0x01010101u * ch;
  const uint32_t a = v.x ^ rep, b = v.y ^ rep, c = v.z ^ rep, d = v.w ^ rep;
  const uint32_t z = ((a - 0x01010101u) & ~a) | ((b - 0x01010101u) & ~b) | ((c - 0x01010101u) & ~c) |
                     ((d - 0x01010101u) & ~d);
  return (z & 0x80808080u) != 0u;
}

// block-wide exclusive scan of one uint32 per thread (blockDim.x multiple of 32, <= 1024).
// `warp_sums` is shared scratch of >= 33 words.  Returns the exclusive prefix; *total gets the block sum.
__device__ __forceinline__ uint32_t block_exclusive_scan(uint32_t v, uint32_t* warp_sums, uint32_t* total) {
  const unsigned lane = lane_id(), warp = threadIdx.x >> 5, nwarps = (blockDim.x + 31) >> 5;
  uint32_t inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= (unsigned)o) inc += t;
  }
  if (lane == 31) warp_sums[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    uint32_t w = lane < nwarps ? warp_sums[lane] : 0;
    uint32_t wi = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      uint32_t t = __shfl_up_sync(0xffffffffu, wi, o);
      if (lane >= (unsigned)o) wi += t;
    }
    if (lane < nwarps) warp_sums[lane] = wi - w;  // exclusive warp offsets
    if (lane == 31) warp_sums[32] = wi;           // block total
  }
  __syncthreads();
  uint32_t r = warp_sums[warp] + inc - v;
  if (total) *total = warp_sums[32];
  __syncthreads();  // scratch may be reused by the caller right away
  return r;
}

__device__ __forceinline__ uint64_t block_exclusive_scan64(uint64_t v, uint64_t* warp_sums, uint64_t* total) {
  const unsigned lane = lane_id(), warp = threadIdx.x >> 5, nwarps = (blockDim.x + 31) >> 5;
  uint64_t inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    uint64_t t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= (unsigned)o) inc += t;
  }
  if (lane == 31) warp_sums[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    uint64_t w = lane < nwarps ? warp_sums[lane] : 0;
    uint64_t wi = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      uint64_t t = __shfl_up_sync(0xffffffffu, wi, o);
      if (lane >= (unsigned)o) wi += t;
    }
    if (lane < nwarps) warp_sums[lane] = wi - w;
    if (lane == 31) warp_sums[32] = wi;
  }
  __syncthreads();
  uint64_t r = warp_sums[warp] + inc - v;
  if (total) *total = warp_sums[32];
  __syncthreads();
  return r;
}

#endif  // __CUDACC__

// ---------------------------------------------------------------------------------------------
// host side of the calls over one dictionary (match.cu, numbers.cu)
// ---------------------------------------------------------------------------------------------
// n host bytes into a fresh device buffer (16 bytes of slack), through the pinned staging arena
inline int upload_host(Ctx* ctx, DevBuf& d, const void* src, size_t n, const char* who) {
  ZDWB_TRY(d.alloc(ctx, n + 16));
  if (!n) return ZDWB_OK;
  void* pinned = stage_take(ctx, n);
  if (!pinned) {
    ctx->err = std::string(who) + ": pinned staging allocation failed";
    return ZDWB_ERR_OOM;
  }
  memcpy(pinned, src, n);
  ZDWB_CUDA_TRY(ctx, cudaMemcpyAsync(d.p, pinned, n, cudaMemcpyHostToDevice, ctx->stream));
  return ZDWB_OK;
}

// the pointer rules of a dictionary given as a zdwb_code_part (its offsets are checked on the device)
inline int check_dict(Ctx* ctx, const zdwb_code_part* d, const char* who) {
  if (!d) {
    ctx->err = std::string(who) + ": dict is NULL";
    return ZDWB_ERR_BAD_ARG;
  }
  if (d->entries > 0 && (!d->dict || !d->entry_off)) {
    ctx->err = std::string(who) + ": entries > 0 with a NULL dict or entry_off";
    return ZDWB_ERR_BAD_ARG;
  }
  return ZDWB_OK;
}

// the call's one host round trip: a small device struct (fault words, totals) copied out once the stream has finished
template <typename T>
int read_back(Ctx* ctx, const void* dev, T* h) {
  ZDWB_CUDA_TRY(ctx, cudaMemcpyAsync(ctx->meta_host, dev, sizeof(T), cudaMemcpyDeviceToHost, ctx->stream));
  ZDWB_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  memcpy(h, ctx->meta_host, sizeof(T));
  return ZDWB_OK;
}

// ---------------------------------------------------------------------------------------------
// generic device-wide primitives (scan.cu / sort.cu)
// ---------------------------------------------------------------------------------------------
// out[i] = sum(in[0..i)), i in [0,n); total (device pointer, may be null) = sum(in[0..n)).  in == out allowed.
int exclusive_scan_u32(Ctx* ctx, const uint32_t* in, uint32_t* out, size_t n, uint32_t* total_dev);
int exclusive_scan_u64(Ctx* ctx, const uint64_t* in, uint64_t* out, size_t n, uint64_t* total_dev);

// Sorts the unique strings of a block into strcmp (unsigned byte, prefix-first) order.
//   base       : device pointer the (start,len) pairs refer to (the TSV buffer)
//   starts/lens: n entries describing each distinct string (no two equal, none containing NUL)
//   order_out  : n entries; order_out[i] = index of the i-th smallest string
int sort_strings(Ctx* ctx, const uint8_t* base, const uint32_t* starts, const uint32_t* lens, uint32_t n,
                 uint32_t max_len, uint32_t* order_out);

}  // namespace zdwb
