// match.cu -- predicates over a sorted dictionary: zdwb_match_like (SQL LIKE, one flag per entry) and zdwb_find_strings
// (lower_bound of query strings).  A dictionary holds each distinct string once, so a filter on a text column costs one
// pass over its dictionary plus one gather per row (zdw_b200/predicates.py).
//
// Kernels (DESIGN 4.8):
//   k_like_match   one thread per entry, plus one for the caller's null text: offsets checked, then the compiled pattern
//   k_find_check   one thread per entry: offsets checked, 16-byte prefix key stored, strictly greater than its
//                  predecessor; one thread per query: offsets checked
//   k_find_search  one thread per query: binary search over the prefix keys, string bytes read only past byte 16; does
//                  nothing when k_find_check found a fault
// Nothing is read through an offset before it has been checked, so garbage input cannot fault the GPU.
#include "common.cuh"

namespace zdwb {

namespace {

constexpr int MT_THREADS = 256;
constexpr uint16_t LIKE_ANY = 256;  // a pattern element that matches any one byte ('_')
constexpr unsigned long long MT_NONE = ~0ull;

// A compiled LIKE pattern: the pattern split at its unescaped '%' into nseg segments; segment s is el[seg[s] .. seg[s+1]),
// each element a literal byte (folded to lower case under ignore_case) or LIKE_ANY.  One segment: no '%' at all.
struct LikePat {
  const uint16_t* el;
  const uint32_t* seg;
  uint32_t nseg;
  uint32_t ignore_case;
};

struct FindMeta {
  unsigned long long ent_err;  // lowest faulty entry << 1 | (0: offsets, 1: order), MT_NONE if none
  unsigned long long q_err;    // lowest query with bad offsets, MT_NONE if none
};

__device__ __forceinline__ unsigned long long grid_threads() { return (unsigned long long)gridDim.x * blockDim.x; }
__device__ __forceinline__ unsigned long long thread_index() { return (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; }

__device__ __forceinline__ uint32_t fold(uint32_t c, uint32_t ic) { return ic && c - 'A' < 26u ? c + 32u : c; }

// segment s at p[0 .. its length)
__device__ __forceinline__ bool seg_at(const LikePat& pat, uint32_t s, const uint8_t* p) {
  const uint32_t a = __ldg(pat.seg + s), b = __ldg(pat.seg + s + 1);
  for (uint32_t i = a; i < b; ++i) {
    const uint32_t e = __ldg(pat.el + i);
    if (e != LIKE_ANY && fold(__ldg(p + (i - a)), pat.ignore_case) != e) return false;
  }
  return true;
}

// LIKE over the whole of p[0 .. L): the first segment anchored at the start, the last at the end, every middle segment
// found leftmost-first behind the one before.  Every segment has a fixed length, so the leftmost place of each leaves
// the most room for the rest: greedy is exact.
__device__ bool like(const LikePat& pat, const uint8_t* p, unsigned long long L) {
  const uint32_t n = pat.nseg;
  const unsigned long long l0 = __ldg(pat.seg + 1) - __ldg(pat.seg);
  if (n == 1) return L == l0 && seg_at(pat, 0, p);
  const unsigned long long ll = __ldg(pat.seg + n) - __ldg(pat.seg + n - 1);
  if (l0 + ll > L || !seg_at(pat, 0, p) || !seg_at(pat, n - 1, p + (L - ll))) return false;
  unsigned long long pos = l0;
  const unsigned long long end = L - ll;
  for (uint32_t s = 1; s + 1 < n; ++s) {
    const unsigned long long ls = __ldg(pat.seg + s + 1) - __ldg(pat.seg + s);
    if (ls == 0) continue;
    for (;; ++pos) {
      if (pos + ls > end) return false;
      if (seg_at(pat, s, p + pos)) break;
    }
    pos += ls;
  }
  return true;
}

// flags[e] = LIKE(entry e) for e < E, flags[E] = LIKE(null text); an entry with bad offsets gets 0 and is reported
__global__ void __launch_bounds__(MT_THREADS)
    k_like_match(const uint8_t* __restrict__ dict, const uint64_t* __restrict__ entry_off, unsigned long long E,
                 unsigned long long dict_bytes, const uint8_t* __restrict__ null_text, unsigned long long null_len, LikePat pat,
                 uint8_t* __restrict__ flags, unsigned long long* __restrict__ bad) {
  for (unsigned long long e = thread_index(); e <= E; e += grid_threads()) {
    const uint8_t* p = null_text;
    unsigned long long L = null_len;
    if (e < E) {
      const unsigned long long a = entry_off[e], b = entry_off[e + 1];
      if (!(a < b && b <= dict_bytes)) {
        atomicMin(bad, e);
        flags[e] = 0;
        continue;
      }
      p = dict + a;
      L = b - a - 1;
    }
    flags[e] = like(pat, p, L) ? 1 : 0;
  }
}

__device__ __forceinline__ ulonglong2 key16(const Str& s) { return make_ulonglong2(key8(s.p, s.len, 0), key8(s.p, s.len, 8)); }

// Entries: offsets, prefix key, order against the predecessor (whose offsets this thread checks as well before it reads
// through them; a fault there is reported by the predecessor's own thread).  Queries: offsets.
__global__ void __launch_bounds__(MT_THREADS)
    k_find_check(const uint8_t* __restrict__ dict, const uint64_t* __restrict__ entry_off, unsigned long long E,
                 unsigned long long dict_bytes, const uint64_t* __restrict__ q_off, unsigned long long n,
                 unsigned long long q_bytes, ulonglong2* __restrict__ keys, FindMeta* meta) {
  const unsigned long long T = E > n ? E : n;
  for (unsigned long long t = thread_index(); t < T; t += grid_threads()) {
    if (t < E) {
      const unsigned long long a = entry_off[t], b = entry_off[t + 1];
      if (!(a < b && b <= dict_bytes)) {
        atomicMin(&meta->ent_err, t << 1);
      } else {
        const Str s{dict + a, b - a - 1};
        const ulonglong2 k = key16(s);
        keys[t] = k;
        if (t > 0) {
          const unsigned long long a0 = entry_off[t - 1];
          if (a0 < a) {
            const Str s0{dict + a0, a - a0 - 1};
            if (str_cmp(key16(s0), s0, k, s) >= 0) atomicMin(&meta->ent_err, t << 1 | 1ull);
          }
        }
      }
    }
    if (t < n) {
      const unsigned long long x = q_off[t], y = q_off[t + 1];
      if (!(x <= y && y <= q_bytes)) atomicMin(&meta->q_err, t);
    }
  }
}

// rank[i] = lower_bound of query i among the entries; found[i] = the entry there equals it
__global__ void __launch_bounds__(MT_THREADS)
    k_find_search(const uint8_t* __restrict__ dict, const uint64_t* __restrict__ entry_off, const ulonglong2* __restrict__ keys,
                  unsigned long long E, const uint8_t* __restrict__ q_bytes, const uint64_t* __restrict__ q_off,
                  unsigned long long n, const FindMeta* __restrict__ meta, long long* __restrict__ rank,
                  uint8_t* __restrict__ found) {
  if (meta->ent_err != MT_NONE || meta->q_err != MT_NONE) return;
  for (unsigned long long i = thread_index(); i < n; i += grid_threads()) {
    const unsigned long long x = q_off[i];
    const Str q{q_bytes + x, q_off[i + 1] - x};
    const ulonglong2 kq = key16(q);
    unsigned long long lo = 0, hi = E;
    bool eq = false;
    while (lo < hi) {
      const unsigned long long mid = (lo + hi) >> 1;
      const ulonglong2 km = keys[mid];
      int c;
      if (km.x != kq.x) c = km.x < kq.x ? -1 : 1;
      else if (km.y != kq.y) c = km.y < kq.y ? -1 : 1;
      else {
        const unsigned long long a = entry_off[mid];
        c = str_cmp(km, Str{dict + a, entry_off[mid + 1] - a - 1}, kq, q);
      }
      if (c < 0) {
        lo = mid + 1;
      } else {
        hi = mid;
        eq |= c == 0;  // entries are distinct: an equal one is the lower bound
      }
    }
    rank[i] = (long long)lo;
    found[i] = eq ? 1 : 0;
  }
}

unsigned grid_for(const Ctx* ctx, unsigned long long threads) {
  const unsigned long long want = (threads + MT_THREADS - 1) / MT_THREADS;
  const unsigned long long cap = (unsigned long long)ctx->sm_count * 16;
  return (unsigned)std::max<unsigned long long>(1, std::min(want, cap));
}

}  // namespace

int match_like_impl(Ctx* ctx, const zdwb_code_part* d, const zdwb_like_opts* o, zdwb_match_out* out) {
  memset(out, 0, sizeof(*out));
  const char* who = "match_like";
  ZDWB_TRY(check_dict(ctx, d, who));
  if ((o->pattern_len && !o->pattern) || (o->null_text_len && !o->null_text)) {
    ctx->err = "match_like: NULL pattern or null_text with a length";
    return ZDWB_ERR_BAD_ARG;
  }
  if (o->escape < -1 || o->escape > 255) {
    ctx->err = "match_like: escape " + std::to_string(o->escape) + " is neither -1 nor a byte";
    return ZDWB_ERR_BAD_ARG;
  }
  if (o->pattern_len >= 0xffffffffull) {
    ctx->err = "match_like: patterns of 2^32 - 1 bytes and more are not supported";
    return ZDWB_ERR_UNSUPPORTED;
  }
  // compile: segments between the unescaped '%'
  std::vector<uint16_t> el;
  std::vector<uint32_t> seg{0u};
  el.reserve(o->pattern_len);
  for (uint64_t i = 0; i < o->pattern_len; ++i) {
    uint32_t c = o->pattern[i];
    if ((int)c == o->escape) {
      if (++i == o->pattern_len) {
        ctx->err = "match_like: the pattern ends in a lone escape byte";
        return ZDWB_ERR_BAD_ARG;
      }
      el.push_back((uint16_t)(o->ignore_case && o->pattern[i] - 'A' < 26u ? o->pattern[i] + 32u : o->pattern[i]));
    } else if (c == '%') {
      seg.push_back((uint32_t)el.size());
    } else if (c == '_') {
      el.push_back(LIKE_ANY);
    } else {
      el.push_back((uint16_t)(o->ignore_case && c - 'A' < 26u ? c + 32u : c));
    }
  }
  seg.push_back((uint32_t)el.size());
  ZDWB_TRY(call_begin(ctx));
  const unsigned long long E = d->entries;
  DevBuf d_el, d_seg, d_null, d_bad;
  ZDWB_TRY(upload_host(ctx, d_el, el.data(), el.size() * 2, who));
  ZDWB_TRY(upload_host(ctx, d_seg, seg.data(), seg.size() * 4, who));
  ZDWB_TRY(upload_host(ctx, d_null, o->null_text, o->null_text_len, who));
  ZDWB_TRY(d_bad.alloc(ctx, 8));
  ZDWB_CUDA_TRY(ctx, cudaMemsetAsync(d_bad.p, 0xff, 8, ctx->stream));
  uint8_t* flags;
  {
    DevBuf fb;
    ZDWB_TRY(fb.alloc(ctx, E + 1));
    flags = static_cast<uint8_t*>(fb.detach());
  }
  const LikePat pat{d_el.as<uint16_t>(), d_seg.as<uint32_t>(), (uint32_t)seg.size() - 1u, o->ignore_case ? 1u : 0u};
  ZDWB_TRY(launch(ctx, "k_like_match", k_like_match, grid_for(ctx, E + 1), MT_THREADS, 0, d->dict, d->entry_off, E, d->dict_bytes,
                  (const uint8_t*)d_null.as<uint8_t>(), (unsigned long long)o->null_text_len, pat, flags,
                  d_bad.as<unsigned long long>()));
  unsigned long long bad;
  ZDWB_TRY(read_back(ctx, d_bad.p, &bad));
  if (bad != MT_NONE) {
    ctx->err = "match_like: entry " + std::to_string(bad) + " has offsets that are not entry_off[e] < entry_off[e+1] <= dict_bytes";
    return ZDWB_ERR_BAD_ARG;
  }
  out->flags = flags;
  out->n = E + 1;
  return ZDWB_OK;
}

int find_strings_impl(Ctx* ctx, const zdwb_code_part* d, const zdwb_strings* q, zdwb_find_out* out) {
  memset(out, 0, sizeof(*out));
  ZDWB_TRY(check_dict(ctx, d, "find_strings"));
  if ((q->n && !q->off) || (q->bytes_len && !q->bytes)) {
    ctx->err = "find_strings: NULL query offsets or bytes";
    return ZDWB_ERR_BAD_ARG;
  }
  ZDWB_TRY(call_begin(ctx));
  cudaStream_t st = ctx->stream;
  const unsigned long long E = d->entries, n = q->n;
  DevBuf d_keys, d_meta;
  ZDWB_TRY(d_keys.alloc(ctx, std::max<unsigned long long>(E, 1) * sizeof(ulonglong2)));
  ZDWB_TRY(d_meta.alloc(ctx, sizeof(FindMeta)));
  ZDWB_CUDA_TRY(ctx, cudaMemsetAsync(d_meta.p, 0xff, sizeof(FindMeta), st));
  FindMeta* meta = d_meta.as<FindMeta>();
  long long* rank = nullptr;
  uint8_t* found = nullptr;
  if (n) {
    DevBuf rb, fb;
    ZDWB_TRY(rb.alloc(ctx, n * 8));
    ZDWB_TRY(fb.alloc(ctx, n));
    found = static_cast<uint8_t*>(fb.detach());
    rank = static_cast<long long*>(rb.detach());
  }
  const unsigned long long T = std::max(E, n);
  if (T) {
    ZDWB_TRY(launch(ctx, "k_find_check", k_find_check, grid_for(ctx, T), MT_THREADS, 0, d->dict, d->entry_off, E, d->dict_bytes,
                    q->off, n, q->bytes_len, d_keys.as<ulonglong2>(), meta));
  }
  if (n) {
    ZDWB_TRY(launch(ctx, "k_find_search", k_find_search, grid_for(ctx, n), MT_THREADS, 0, d->dict, d->entry_off,
                    (const ulonglong2*)d_keys.as<ulonglong2>(), E, q->bytes, q->off, n, (const FindMeta*)meta, rank, found));
  }
  FindMeta h;
  ZDWB_TRY(read_back(ctx, meta, &h));
  if (h.ent_err != MT_NONE) {
    ctx->err = "find_strings: entry " + std::to_string(h.ent_err >> 1) +
               ((h.ent_err & 1) ? " is not greater than the entry before it (the entries must be strictly increasing bytewise)"
                                : " has offsets that are not entry_off[e] < entry_off[e+1] <= dict_bytes");
    return ZDWB_ERR_BAD_ARG;
  }
  if (h.q_err != MT_NONE) {
    ctx->err = "find_strings: query " + std::to_string(h.q_err) + " has offsets that are not off[i] <= off[i+1] <= bytes_len";
    return ZDWB_ERR_BAD_ARG;
  }
  out->rank = reinterpret_cast<const int64_t*>(rank);
  out->found = found;
  out->n = n;
  return ZDWB_OK;
}

}  // namespace zdwb
