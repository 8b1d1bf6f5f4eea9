// render.cu -- zdwb_render_columns: typed device columns -> the TSV rows that zdwb_encode_block turns back into the same
// cells.  A file written from columns is then exactly what convertDWfile makes of that text (include/zdw_b200.h).
//
// Kernels, in order (DESIGN 4.7):
//   k_render_entries  one thread per entry of every distinct dictionary: may it be written as a field?  (status byte)
//   k_render_lengths  one thread per row (a warp's 32 cells of a column are one 256-byte load): range checks, the
//                     entries' status, every cell's text length, the row's length
//   (scan)            row lengths -> row offsets and the output size
//   k_render_write    a group of 8, 16 or 32 lanes per row, one cell per lane and step: numbers and short texts by the
//                     lane, texts longer than 16 bytes by the whole group in aligned words
// Nothing is read through an entry's offsets before they have been checked against the dictionary's size.
#include "common.cuh"

namespace zdwb {

namespace {

constexpr int RD_THREADS = 256;
constexpr uint32_t RD_LONG = 16;  // longer texts are copied by the whole group

// a column as the kernels see it
struct RCol {
  const int64_t* codes;
  const uint64_t* entry_off;   // text-like only
  const uint8_t* dict;         // text-like only
  const uint8_t* status;       // text-like only: RD_* per entry of the column's dictionary
  unsigned long long entries;  // text-like only
  uint32_t type;
  uint32_t reserved;
};

// a distinct dictionary
struct RDict {
  const uint8_t* dict;
  const uint64_t* entry_off;
  unsigned long long entries;
  unsigned long long dict_bytes;
};

// rules a cell can break; the error key is column << 40 | row << 4 | rule, so its minimum names the lowest (column, row)
enum : uint32_t {
  RD_OK = 0,
  RD_OFFSETS = 1,   // entry offsets not entry_off[e] < entry_off[e+1] <= dict_bytes
  RD_ENTRY = 2,     // entry empty, NUL inside, or not NUL-terminated
  RD_SEPARATOR = 3, // entry holds a tab or newline that is not escaped by an odd run of backslashes
  RD_BACKSLASH = 4, // entry ends in an odd run of backslashes
  RD_CODE = 5,      // code < -1 or >= entries
  RD_CHAR = 6,      // CHAR value none of the three forms
  RD_EMPTY_ROW = 7, // one column and an empty cell: the row would be "\n"
};
constexpr unsigned long long RD_NO_ERROR = ~0ull;

struct RenderMeta {
  unsigned long long err;    // lowest error key, RD_NO_ERROR if none
  unsigned long long total;  // output bytes
};

__device__ __forceinline__ unsigned long long grid_threads() { return (unsigned long long)gridDim.x * blockDim.x; }
__device__ __forceinline__ unsigned long long thread_index() { return (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; }

// the last i with a[i] <= x (a ascending, a[0] <= x)
__device__ __forceinline__ uint32_t last_le(const unsigned long long* __restrict__ a, uint32_t n, unsigned long long x) {
  uint32_t lo = 0, hi = n;
  while (hi - lo > 1) {
    const uint32_t mid = (lo + hi) >> 1;
    if (a[mid] <= x) lo = mid;
    else hi = mid;
  }
  return lo;
}

// Entry status.  The row reader (oracle next_row / next_column) ends a field at a tab and a row at a newline unless an
// odd run of backslashes stands in front; a field that ends in an odd run escapes the separator behind it.
__global__ void __launch_bounds__(RD_THREADS)
    k_render_entries(const RDict* __restrict__ dicts, const unsigned long long* __restrict__ ent_base, uint32_t D,
                     unsigned long long E, uint8_t* __restrict__ status) {
  for (unsigned long long g = thread_index(); g < E; g += grid_threads()) {
    const uint32_t d = last_le(ent_base, D + 1, g);
    const RDict& rd = dicts[d];
    const unsigned long long e = g - ent_base[d];
    const unsigned long long a = rd.entry_off[e], b = rd.entry_off[e + 1];
    uint32_t st = RD_OK;
    if (!(a < b && b <= rd.dict_bytes)) {
      st = RD_OFFSETS;
    } else if (b - a < 2 || __ldg(rd.dict + b - 1) != 0) {
      st = RD_ENTRY;
    } else {
      uint32_t run = 0;
      for (unsigned long long i = a; i < b - 1; ++i) {
        const uint8_t ch = __ldg(rd.dict + i);
        if (ch == 0) {
          st = RD_ENTRY;
          break;
        }
        if ((ch == '\t' || ch == '\n') && !(run & 1u)) {
          st = RD_SEPARATOR;
          break;
        }
        run = ch == '\\' ? run + 1u : 0u;
      }
      if (st == RD_OK && (run & 1u)) st = RD_BACKSLASH;
    }
    status[g] = (uint8_t)st;
  }
}

// Text length of a number or CHAR cell (rule in *rule when the value has no text that reads back).
__device__ __forceinline__ uint32_t scalar_len(uint32_t t, long long v, uint32_t* rule) {
  if (t == ZDWB_CHAR) {
    if (v == 0) return 0;
    if (v >= -128 && v <= 127) {  // sx(b0): one byte, not NUL, tab, newline or backslash
      if (v == '\t' || v == '\n' || v == '\\') *rule = RD_CHAR;
      return 1;
    }
    const long long k = (v - '\\') >> 8;  // '\\' + sx(b1) * 256, b1 != NUL
    if (((v - '\\') & 255) != 0 || k < -128 || k > 127 || k == 0) *rule = RD_CHAR;
    return 2;
  }
  if (is_signed_int_type((uint8_t)t) && v < 0) return 1u + digits_u64(0ull - (unsigned long long)v);
  return digits_u64((unsigned long long)v);
}

__global__ void __launch_bounds__(RD_THREADS)
    k_render_lengths(const RCol* __restrict__ cols, uint32_t K, unsigned long long n, unsigned long long* __restrict__ row_len,
                     RenderMeta* meta) {
  const unsigned long long r = thread_index();
  if (r >= n) return;
  unsigned long long len = K;  // K - 1 tabs and the newline
  unsigned long long err = RD_NO_ERROR;
  for (uint32_t k = 0; k < K && err == RD_NO_ERROR; ++k) {
    const uint32_t t = cols[k].type;
    const long long v = __ldg(cols[k].codes + r);
    uint32_t rule = RD_OK, l = 0;
    if (is_text_like((uint8_t)t)) {
      if (v != -1) {
        if (v < -1 || (unsigned long long)v >= cols[k].entries) {
          rule = RD_CODE;
        } else {
          rule = __ldg(cols[k].status + v);
          if (rule == RD_OK) l = (uint32_t)(__ldg(cols[k].entry_off + v + 1) - __ldg(cols[k].entry_off + v) - 1);
        }
      }
    } else {
      l = scalar_len(t, v, &rule);
    }
    if (rule == RD_OK && l == 0 && K == 1) rule = RD_EMPTY_ROW;
    if (rule != RD_OK) err = ((unsigned long long)k << 40) | (r << 4) | rule;
    len += l;
  }
  if (err != RD_NO_ERROR) atomicMin(&meta->err, err);
  row_len[r] = len;
}

// n bytes from s to d by the G lanes of a group: head bytes up to d's next 4-byte boundary (lane 0), aligned words
// funnel-shifted out of two aligned source words (one per lane and step), tail bytes (lane 1) -- decode.cu's octet_copy
// for any group width
template <int G>
__device__ __forceinline__ void group_copy(uint8_t* __restrict__ d, const uint8_t* __restrict__ s, uint32_t n, unsigned gl) {
  const uint32_t head = min(n, (4u - (uint32_t)(reinterpret_cast<uintptr_t>(d) & 3u)) & 3u);
  if (gl == 0) {
    for (uint32_t k = 0; k < head; ++k) d[k] = __ldg(s + k);
  }
  const uint32_t nw = (n - head) >> 2, tail = (n - head) & 3u;
  const uintptr_t a = reinterpret_cast<uintptr_t>(s + head);
  const uint32_t* w = reinterpret_cast<const uint32_t*>(a & ~(uintptr_t)3);
  const uint32_t sh = (uint32_t)(a & 3u) * 8u;
  uint32_t* dw = reinterpret_cast<uint32_t*>(d + head);
  for (uint32_t k = gl; k < nw; k += G) {
    const uint32_t lo = __ldg(w + k);
    const uint32_t hi = sh ? __ldg(w + k + 1) : 0u;
    dw[k] = __funnelshift_r(lo, hi, sh);
  }
  if (gl == 1) {
    for (uint32_t k = 0; k < tail; ++k) d[head + 4u * nw + k] = __ldg(s + head + 4u * nw + k);
  }
}

// One group of G lanes per row; lane j of a step writes cell k0 + j and the separator behind it.  Every input has
// passed k_render_lengths.
template <int G>
__global__ void __launch_bounds__(RD_THREADS)
    k_render_write(const RCol* __restrict__ cols, uint32_t K, unsigned long long n, const unsigned long long* __restrict__ row_off,
                   uint8_t* __restrict__ out) {
  constexpr uint32_t GPW = 32 / G;
  const unsigned lane = lane_id(), gl = lane & (unsigned)(G - 1);
  const unsigned gm = G == 32 ? 0xffffffffu : (((1u << G) - 1u) << (lane & ~(unsigned)(G - 1)));
  const unsigned long long groups = grid_threads() / G;
  for (unsigned long long r = thread_index() / G; r < n; r += groups) {
    uint8_t* row = out + row_off[r];
    unsigned long long at = 0;  // bytes of the row written by the steps before
    for (uint32_t k0 = 0; k0 < K; k0 += G) {
      const uint32_t k = k0 + gl;
      uint32_t l = 0, w[5] = {0u, 0u, 0u, 0u, 0u};
      const uint8_t* src = nullptr;
      if (k < K) {
        const uint32_t t = cols[k].type;
        const long long v = __ldg(cols[k].codes + r);
        if (is_text_like((uint8_t)t)) {
          if (v >= 0) {
            const unsigned long long a = __ldg(cols[k].entry_off + v);
            l = (uint32_t)(__ldg(cols[k].entry_off + v + 1) - a - 1);
            src = cols[k].dict + a;
          }
        } else if (t == ZDWB_CHAR) {
          l = v == 0 ? 0u : ((v & 255) == '\\' ? 2u : 1u);
          w[0] = (uint32_t)v & 0xffffu;
        } else {
          uint32_t rule = RD_OK;
          l = scalar_len(t, v, &rule);
          const bool neg = is_signed_int_type((uint8_t)t) && v < 0;
          if (neg && v == (long long)0x8000000000000000ull) {
            // render_int keeps lltoa's digits for INT64_MIN, which do not parse back: the plain text instead
            w[0] = 0x3232392du;  // "-922"
            w[1] = 0x32373333u;  // "3372"
            w[2] = 0x38363330u;  // "0368"
            w[3] = 0x37373435u;  // "5477"
            w[4] = 0x38303835u;  // "5808"
          } else {
            render_int((unsigned long long)v, neg, l, w);
          }
        }
      }
      // offsets of the cells of this step: inclusive scan of (length + separator) over the group
      uint32_t inc = k < K ? l + 1u : 0u;
#pragma unroll
      for (int o = 1; o < G; o <<= 1) {
        const uint32_t x = __shfl_up_sync(gm, inc, o, G);
        if (gl >= (unsigned)o) inc += x;
      }
      const uint32_t step = __shfl_sync(gm, inc, G - 1, G);
      uint8_t* d = row + at + (inc - (k < K ? l + 1u : 0u));
      if (k < K) {
        if (src == nullptr || l <= RD_LONG) {
          if (src) {
            for (uint32_t i = 0; i < l; ++i) d[i] = __ldg(src + i);
          } else {
            for (uint32_t i = 0; i < l; ++i) d[i] = (uint8_t)(w[i >> 2] >> ((i & 3u) * 8u));
          }
        }
        d[l] = k + 1 == K ? '\n' : '\t';
      }
      // long texts: the whole group copies each in turn
      unsigned long_lanes = __ballot_sync(gm, src != nullptr && l > RD_LONG) >> (lane & ~(unsigned)(G - 1));
      if (G < 32) long_lanes &= (1u << G) - 1u;
      while (long_lanes) {
        const unsigned j = (unsigned)__ffs(long_lanes) - 1u;
        long_lanes &= long_lanes - 1u;
        const unsigned long long dj = __shfl_sync(gm, (unsigned long long)(d - out), j, G);
        const unsigned long long sj = __shfl_sync(gm, (unsigned long long)reinterpret_cast<uintptr_t>(src), j, G);
        const uint32_t lj = __shfl_sync(gm, l, j, G);
        group_copy<G>(out + dj, reinterpret_cast<const uint8_t*>(sj), lj, gl);
      }
      at += step;
    }
  }
}

unsigned grid_for(const Ctx* ctx, unsigned long long threads) {
  const unsigned long long want = (threads + RD_THREADS - 1) / RD_THREADS;
  const unsigned long long cap = (unsigned long long)ctx->sm_count * 16;
  return (unsigned)std::max<unsigned long long>(1, std::min(want, cap));
}

template <typename T>
int render_upload(Ctx* ctx, DevBuf& d, const std::vector<T>& v) {
  const size_t n = v.size() * sizeof(T);
  ZDWB_TRY(d.alloc(ctx, n + 16));
  void* pinned = stage_take(ctx, n);
  if (!pinned) {
    ctx->err = "render_columns: pinned staging allocation failed";
    return ZDWB_ERR_OOM;
  }
  memcpy(pinned, v.data(), n);
  ZDWB_CUDA_TRY(ctx, cudaMemcpyAsync(d.p, pinned, n, cudaMemcpyHostToDevice, ctx->stream));
  return ZDWB_OK;
}

const char* rule_text(uint32_t rule) {
  switch (rule) {
    case RD_OFFSETS: return "references an entry whose offsets are not entry_off[e] < entry_off[e+1] <= dict_bytes";
    case RD_ENTRY: return "references an entry that is empty, holds a NUL or does not end in a NUL";
    case RD_SEPARATOR: return "references an entry with a tab or newline not escaped by an odd run of backslashes";
    case RD_BACKSLASH: return "references an entry that ends in an odd run of backslashes";
    case RD_CODE: return "holds a code < -1 or >= its number of entries";
    case RD_CHAR: return "holds a CHAR value that is not 0, sx(b) for b not NUL, tab, newline or backslash, or '\\\\' + sx(b) * 256 for b not NUL";
    case RD_EMPTY_ROW: return "renders empty in a table of one column (the row would be skipped)";
    default: return "is invalid";
  }
}

}  // namespace

int render_columns_impl(Ctx* ctx, const zdwb_schema* schema, const zdwb_code_part* cols, void** buf, size_t* cap,
                        zdwb_render_out* out) {
  memset(out, 0, sizeof(*out));
  if (!schema->types || !cols) {
    ctx->err = "render_columns: NULL types or columns";
    return ZDWB_ERR_BAD_ARG;
  }
  const uint32_t K = schema->ncols;
  if (K == 0) {
    ctx->err = "render_columns: zero columns";
    return ZDWB_ERR_BAD_ARG;
  }
  if (K >= (1u << 24)) {
    ctx->err = "render_columns: more than 2^24 - 1 columns";
    return ZDWB_ERR_UNSUPPORTED;
  }
  const unsigned long long n = cols[0].n;
  std::vector<RCol> hc(K);
  std::vector<RDict> hd;
  std::vector<uint32_t> dict_of(K, 0);
  for (uint32_t k = 0; k < K; ++k) {
    const zdwb_code_part& c = cols[k];
    const uint8_t t = schema->types[k];
    if (c.n != n) {
      ctx->err = "render_columns: column " + std::to_string(k) + " has " + std::to_string(c.n) + " rows, column 0 has " +
                 std::to_string(n);
      return ZDWB_ERR_BAD_ARG;
    }
    if (!is_known_type(t)) {
      ctx->err = "render_columns: column " + std::to_string(k) + " has type " + std::to_string(t) + ", which the encoder does not know";
      return ZDWB_ERR_BAD_ARG;
    }
    if (n && !c.codes) {
      ctx->err = "render_columns: column " + std::to_string(k) + " has rows but a NULL codes pointer";
      return ZDWB_ERR_BAD_ARG;
    }
    hc[k] = RCol{c.codes, nullptr, nullptr, nullptr, 0ull, t, 0u};
    if (is_text_like(t)) {
      if (c.entries > 0 && (!c.dict || !c.entry_off)) {
        ctx->err = "render_columns: column " + std::to_string(k) + " has entries but a NULL dict or entry_off";
        return ZDWB_ERR_BAD_ARG;
      }
      hc[k].entry_off = c.entry_off;
      hc[k].dict = c.dict;
      hc[k].entries = c.entries;
      uint32_t d = 0;  // columns that share a dictionary share its status bytes
      while (d < hd.size() && !(hd[d].dict == c.dict && hd[d].entry_off == c.entry_off && hd[d].entries == c.entries &&
                                hd[d].dict_bytes == c.dict_bytes))
        ++d;
      if (d == hd.size()) hd.push_back(RDict{c.dict, c.entry_off, c.entries, c.dict_bytes});
      dict_of[k] = d;
    }
  }
  if (n >= (1ull << 36)) {
    ctx->err = "render_columns: more than 2^36 - 1 rows";
    return ZDWB_ERR_UNSUPPORTED;
  }
  ZDWB_TRY(call_begin(ctx));
  if (n == 0) {
    out->tsv = static_cast<const uint8_t*>(*buf);
    return ZDWB_OK;
  }
  cudaStream_t st = ctx->stream;
  const uint32_t D = (uint32_t)hd.size();
  std::vector<unsigned long long> ent_base(D + 1, 0);
  for (uint32_t d = 0; d < D; ++d) ent_base[d + 1] = ent_base[d] + hd[d].entries;
  const unsigned long long E = ent_base[D];

  DevBuf d_status, d_dicts, d_ent_base, d_cols, d_meta, d_len;
  ZDWB_TRY(d_status.alloc(ctx, E + 16));
  uint8_t* status = d_status.as<uint8_t>();
  for (uint32_t k = 0; k < K; ++k)
    if (is_text_like(schema->types[k])) hc[k].status = status + ent_base[dict_of[k]];
  ZDWB_TRY(render_upload(ctx, d_cols, hc));
  ZDWB_TRY(d_meta.alloc(ctx, sizeof(RenderMeta)));
  ZDWB_CUDA_TRY(ctx, cudaMemsetAsync(d_meta.p, 0xff, sizeof(RenderMeta), st));
  RenderMeta* meta = d_meta.as<RenderMeta>();
  if (E) {
    ZDWB_TRY(render_upload(ctx, d_dicts, hd));
    ZDWB_TRY(render_upload(ctx, d_ent_base, ent_base));
    ZDWB_TRY(launch(ctx, "k_render_entries", k_render_entries, grid_for(ctx, E), RD_THREADS, 0, (const RDict*)d_dicts.as<RDict>(),
                    (const unsigned long long*)d_ent_base.as<unsigned long long>(), D, E, status));
  }
  const RCol* dcols = d_cols.as<RCol>();
  ZDWB_TRY(d_len.alloc(ctx, (n + 1) * 8));
  unsigned long long* row_len = d_len.as<unsigned long long>();
  ZDWB_TRY(launch(ctx, "k_render_lengths", k_render_lengths, (unsigned)((n + RD_THREADS - 1) / RD_THREADS), RD_THREADS, 0, dcols, K,
                  n, row_len, meta));
  ZDWB_TRY(exclusive_scan_u64(ctx, reinterpret_cast<uint64_t*>(row_len), reinterpret_cast<uint64_t*>(row_len), n,
                              reinterpret_cast<uint64_t*>(&meta->total)));
  ZDWB_CUDA_TRY(ctx, cudaMemcpyAsync(ctx->meta_host, meta, sizeof(RenderMeta), cudaMemcpyDeviceToHost, st));
  ZDWB_CUDA_TRY(ctx, cudaStreamSynchronize(st));
  RenderMeta h;
  memcpy(&h, ctx->meta_host, sizeof(h));
  if (h.err != RD_NO_ERROR) {
    const unsigned long long col = h.err >> 40, row = (h.err >> 4) & ((1ull << 36) - 1);
    ctx->err = "render_columns: column " + std::to_string(col) + " row " + std::to_string(row) + " " + rule_text((uint32_t)(h.err & 15u));
    return ZDWB_ERR_BAD_ARG;
  }

  // the output buffer is the context's own allocation: it outlives the arena resets of the calls that follow
  if (*cap < h.total + 16) {
    ZDWB_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));  // (an encode of the previous rendering may still read it)
    if (*buf) cudaFree(*buf);
    *buf = nullptr;
    *cap = 0;
    const size_t want = h.total + h.total / 8 + 64;  // headroom: the blocks of a file vary a little
    ZDWB_CUDA_TRY(ctx, cudaMalloc(buf, want));
    *cap = want;
  }
  uint8_t* dst = static_cast<uint8_t*>(*buf);
  if (K <= 8) {
    ZDWB_TRY(launch(ctx, "k_render_write", k_render_write<8>, grid_for(ctx, n * 8), RD_THREADS, 0, dcols, K, n,
                    (const unsigned long long*)row_len, dst));
  } else if (K <= 16) {
    ZDWB_TRY(launch(ctx, "k_render_write", k_render_write<16>, grid_for(ctx, n * 16), RD_THREADS, 0, dcols, K, n,
                    (const unsigned long long*)row_len, dst));
  } else {
    ZDWB_TRY(launch(ctx, "k_render_write", k_render_write<32>, grid_for(ctx, n * 32), RD_THREADS, 0, dcols, K, n,
                    (const unsigned long long*)row_len, dst));
  }
  ZDWB_CUDA_TRY(ctx, cudaStreamSynchronize(st));
  out->tsv = dst;
  out->len = h.total;
  return ZDWB_OK;
}

}  // namespace zdwb
