// numbers.cu -- DATETIME and DECIMAL dictionary strings as numbers and back: zdwb_parse_numbers (one number per entry)
// and zdwb_format_numbers (strictly increasing numbers -> a dense, sorted dictionary and their codes into it).  A
// dictionary holds each distinct string once, so a conversion of a column costs one pass over its distinct strings plus
// one gather per row (zdw_b200/numbers.py).
//
// Kernels (DESIGN 4.9):
//   k_num_parse    one thread per entry, plus one for the caller's null text: offsets checked, then the text parsed
//   k_num_check    one thread per value: order against the predecessor, range, exactness; the text's length + 1
//   (scan)         lengths -> where each text goes in a scratch buffer
//   k_num_write    one thread per value: its text, NUL-terminated, and the (start, length) the string sort takes
//   (sort_strings) the bytewise order of the texts
//   k_num_sorted_lens, (scan), k_num_emit   the dictionary in that order, its entry offsets and the codes
// Nothing is read through an offset before it has been checked, so garbage input cannot fault the GPU.
#include "common.cuh"

namespace zdwb {

namespace {

constexpr int NM_THREADS = 256;
constexpr unsigned long long NM_NONE = ~0ull;
constexpr long long US_PER_DAY = 86400000000ll;
// format faults, the low two bits of the fault word (value << 2 | kind): the lowest value wins, then the lowest kind
constexpr unsigned long long NM_ORDER = 0, NM_RANGE = 1, NM_INEXACT = 2;

__constant__ unsigned long long kPow10[20] = {1ull, 10ull, 100ull, 1000ull, 10000ull, 100000ull, 1000000ull, 10000000ull,
                                              100000000ull, 1000000000ull, 10000000000ull, 100000000000ull,
                                              1000000000000ull, 10000000000000ull, 100000000000000ull,
                                              1000000000000000ull, 10000000000000000ull, 100000000000000000ull,
                                              1000000000000000000ull, 10000000000000000000ull};

struct FormatMeta {
  unsigned long long bad;    // lowest value at fault << 2 | NM_*, NM_NONE if none
  unsigned long long total;  // sum over the values of (text length + 1)
};

__device__ __forceinline__ unsigned long long grid_threads() { return (unsigned long long)gridDim.x * blockDim.x; }
__device__ __forceinline__ unsigned long long thread_index() { return (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; }

// days from 1970-01-01 to y-m-d on the proleptic Gregorian calendar, closed form (eras of 400 years, March-based years)
__host__ __device__ __forceinline__ long long days_from_civil(long long y, unsigned m, unsigned d) {
  y -= m <= 2;
  const long long era = (y >= 0 ? y : y - 399) / 400;
  const unsigned yoe = (unsigned)(y - era * 400);
  const unsigned doy = (153u * (m > 2 ? m - 3 : m + 9) + 2u) / 5u + d - 1u;
  const unsigned doe = yoe * 365u + yoe / 4u - yoe / 100u + doy;
  return era * 146097 + (long long)doe - 719468;
}

// the inverse of days_from_civil
__device__ __forceinline__ void civil_from_days(long long z, long long* y, unsigned* m, unsigned* d) {
  z += 719468;
  const long long era = (z >= 0 ? z : z - 146096) / 146097;
  const unsigned doe = (unsigned)(z - era * 146097);
  const unsigned yoe = (doe - doe / 1460u + doe / 36524u - doe / 146096u) / 365u;
  const unsigned doy = doe - (365u * yoe + yoe / 4u - yoe / 100u);
  const unsigned mp = (5u * doy + 2u) / 153u;
  *d = doy - (153u * mp + 2u) / 5u + 1u;
  *m = mp < 10u ? mp + 3u : mp - 9u;
  *y = (long long)yoe + era * 400 + (*m <= 2u);
}

constexpr long long DT_MIN = -62135596800000000ll;                  // 0001-01-01 00:00:00
constexpr long long DT_MAX = 253402300800000000ll - 1ll;            // 9999-12-31 23:59:59.999999
static_assert(DT_MIN == -719162ll * US_PER_DAY, "0001-01-01 is day -719162");
static_assert(DT_MAX + 1 == 2932897ll * US_PER_DAY, "10000-01-01 is day 2932897");

// n digits at p (n <= 6); *ok cleared when one of them is not a digit
__device__ __forceinline__ unsigned digits_at(const uint8_t* p, int n, bool* ok) {
  unsigned v = 0;
  for (int i = 0; i < n; ++i) {
    const unsigned c = (unsigned)__ldg(p + i) - '0';
    *ok &= c < 10u;
    v = v * 10u + c;
  }
  return v;
}

// "YYYY-MM-DD[ HH:MM:SS[.F{1,6}]]" -> microseconds since 1970-01-01; false when the text is not one or the date or
// time does not exist.  Lengths other than 10, 19 and 21..26 are refused before a byte is read.
__device__ bool parse_datetime(const uint8_t* p, unsigned long long L, long long* v) {
  if (!(L == 10 || L == 19 || (L >= 21 && L <= 26))) return false;
  bool ok = __ldg(p + 4) == '-' && __ldg(p + 7) == '-';
  const unsigned y = digits_at(p, 4, &ok), mo = digits_at(p + 5, 2, &ok), d = digits_at(p + 8, 2, &ok);
  unsigned h = 0, mi = 0, s = 0, us = 0;
  if (L > 10) {
    ok &= __ldg(p + 10) == ' ' && __ldg(p + 13) == ':' && __ldg(p + 16) == ':';
    h = digits_at(p + 11, 2, &ok);
    mi = digits_at(p + 14, 2, &ok);
    s = digits_at(p + 17, 2, &ok);
  }
  if (L > 19) {
    const int nf = (int)L - 20;
    ok &= __ldg(p + 19) == '.';
    us = digits_at(p + 20, nf, &ok) * (unsigned)kPow10[6 - nf];
  }
  if (!ok || y == 0 || mo - 1u >= 12u || d == 0 || h > 23u || mi > 59u || s > 59u) return false;
  const bool leap = y % 4u == 0 && (y % 100u != 0 || y % 400u == 0);
  const unsigned mdays = mo == 2 ? 28u + leap : 30u + ((0x15AAu >> mo) & 1u);  // 31 in months 1 3 5 7 8 10 12
  if (d > mdays) return false;
  *v = days_from_civil(y, mo, d) * US_PER_DAY + (long long)(h * 3600u + mi * 60u + s) * 1000000ll + us;
  return true;
}

// [+-]?(D+(\.D*)?|\.D+) times 10^s, exact and within int64 -> *v; false otherwise.  One walk that stops at the first
// byte outside the grammar; the magnitude is accumulated in uint64 against 2^63, the sign applied last.
__device__ bool parse_decimal(const uint8_t* p, unsigned long long L, uint32_t s, long long* v) {
  constexpr unsigned long long LIM = 1ull << 63;
  unsigned long long i = 0, m = 0;
  bool neg = false, dot = false;
  uint32_t nd = 0, fd = 0;  // digits seen; fraction digits taken into m
  if (L) {
    const uint8_t c = __ldg(p);
    if (c == '+' || c == '-') {
      neg = c == '-';
      i = 1;
    }
  }
  for (; i < L; ++i) {
    const uint8_t c = __ldg(p + i);
    if (c == '.') {
      if (dot) return false;
      dot = true;
      continue;
    }
    const unsigned dg = (unsigned)c - '0';
    if (dg > 9u) return false;
    ++nd;
    if (dot) {
      if (fd == s) {
        if (dg) return false;  // not exact at this scale
        continue;
      }
      ++fd;
    }
    if (m > (LIM - dg) / 10u) return false;
    m = m * 10u + dg;
  }
  if (nd == 0) return false;
  for (; fd < s; ++fd) {
    if (m > LIM / 10u) return false;
    m *= 10u;
  }
  if (!neg && m == LIM) return false;
  *v = (long long)(neg ? 0ull - m : m);
  return true;
}

// values[e], ok[e] of entry e < E, and of the null text at e == E; an entry with bad offsets gets 0, 0 and is reported
__global__ void __launch_bounds__(NM_THREADS)
    k_num_parse(const uint8_t* __restrict__ dict, const uint64_t* __restrict__ entry_off, unsigned long long E,
                unsigned long long dict_bytes, const uint8_t* __restrict__ null_text, unsigned long long null_len, int kind,
                uint32_t scale, long long* __restrict__ values, uint8_t* __restrict__ ok, unsigned long long* __restrict__ bad) {
  for (unsigned long long e = thread_index(); e <= E; e += grid_threads()) {
    const uint8_t* p = null_text;
    unsigned long long L = null_len;
    if (e < E) {
      const unsigned long long a = entry_off[e], b = entry_off[e + 1];
      if (!(a < b && b <= dict_bytes)) {
        atomicMin(bad, e);
        values[e] = 0;
        ok[e] = 0;
        continue;
      }
      p = dict + a;
      L = b - a - 1;
    }
    long long v = 0;
    const bool good = kind == ZDWB_NUM_DATETIME ? parse_datetime(p, L, &v) : parse_decimal(p, L, scale, &v);
    values[e] = good ? v : 0;
    ok[e] = good ? 1 : 0;
  }
}

// the text of v: 19 + (digits ? 1 + digits : 0) bytes for DATETIME, sign + integer digits + (digits ? 1 + digits : 0)
// for DECIMAL
__device__ __forceinline__ uint32_t text_len(int kind, uint32_t digits, long long v) {
  const uint32_t frac = digits ? 1u + digits : 0u;
  if (kind == ZDWB_NUM_DATETIME) return 19u + frac;
  const unsigned long long m = v < 0 ? 0ull - (unsigned long long)v : (unsigned long long)v;
  return (v < 0 ? 1u : 0u) + digits_u64(m / kPow10[digits]) + frac;
}

// n digits of x, zero-padded, ending at q[n - 1]
__device__ __forceinline__ void put_digits(uint8_t* q, uint32_t n, unsigned long long x) {
  for (uint32_t i = n; i-- > 0;) {
    q[i] = (uint8_t)('0' + x % 10u);
    x /= 10u;
  }
}

// writes the text of v (text_len bytes) at q
__device__ void write_text(int kind, uint32_t digits, long long v, uint8_t* q) {
  if (kind == ZDWB_NUM_DATETIME) {
    long long days = v / US_PER_DAY, rem = v % US_PER_DAY;
    if (rem < 0) {
      rem += US_PER_DAY;
      --days;
    }
    long long y;
    unsigned mo, d;
    civil_from_days(days, &y, &mo, &d);
    const unsigned secs = (unsigned)(rem / 1000000), us = (unsigned)(rem % 1000000);
    put_digits(q, 4, (unsigned long long)y);
    q[4] = '-';
    put_digits(q + 5, 2, mo);
    q[7] = '-';
    put_digits(q + 8, 2, d);
    q[10] = ' ';
    put_digits(q + 11, 2, secs / 3600u);
    q[13] = ':';
    put_digits(q + 14, 2, secs / 60u % 60u);
    q[16] = ':';
    put_digits(q + 17, 2, secs % 60u);
    if (digits) {
      q[19] = '.';
      put_digits(q + 20, digits, us / kPow10[6 - digits]);
    }
    return;
  }
  const unsigned long long m = v < 0 ? 0ull - (unsigned long long)v : (unsigned long long)v;
  const unsigned long long ip = m / kPow10[digits];
  if (v < 0) *q++ = '-';
  const uint32_t ni = digits_u64(ip);
  put_digits(q, ni, ip);
  if (digits) {
    q[ni] = '.';
    put_digits(q + ni + 1, digits, m % kPow10[digits]);
  }
}

// per value: order against its predecessor, DATETIME range and exactness; lens[i] = text length + 1
__global__ void __launch_bounds__(NM_THREADS)
    k_num_check(const long long* __restrict__ values, unsigned long long n, int kind, uint32_t digits,
                unsigned long long* __restrict__ lens, FormatMeta* meta) {
  for (unsigned long long i = thread_index(); i < n; i += grid_threads()) {
    const long long v = values[i];
    if (i > 0 && values[i - 1] >= v) atomicMin(&meta->bad, i << 2 | NM_ORDER);
    if (kind == ZDWB_NUM_DATETIME) {
      if (v < DT_MIN || v > DT_MAX) atomicMin(&meta->bad, i << 2 | NM_RANGE);
      else if (v % (long long)kPow10[6 - digits] != 0) atomicMin(&meta->bad, i << 2 | NM_INEXACT);
    }
    lens[i] = text_len(kind, digits, v) + 1u;
  }
}

// the text of value i at text + off[i], NUL-terminated; its (start, length) for the string sort
__global__ void __launch_bounds__(NM_THREADS)
    k_num_write(const long long* __restrict__ values, unsigned long long n, int kind, uint32_t digits,
                const unsigned long long* __restrict__ off, uint8_t* __restrict__ text, uint32_t* __restrict__ starts,
                uint32_t* __restrict__ lens) {
  for (unsigned long long i = thread_index(); i < n; i += grid_threads()) {
    const long long v = values[i];
    const unsigned long long o = off[i];
    const uint32_t L = text_len(kind, digits, v);
    write_text(kind, digits, v, text + o);
    text[o + L] = 0;
    starts[i] = (uint32_t)o;
    lens[i] = L;
  }
}

__global__ void __launch_bounds__(NM_THREADS)
    k_num_sorted_lens(const uint32_t* __restrict__ order, const uint32_t* __restrict__ lens, unsigned long long n,
                      unsigned long long* __restrict__ entry_off) {
  for (unsigned long long j = thread_index(); j < n; j += grid_threads()) entry_off[j] = lens[order[j]] + 1ull;
}

// entry j of the dictionary is text order[j]: its bytes behind the origin NUL, its offset, and codes[order[j]] = j
__global__ void __launch_bounds__(NM_THREADS)
    k_num_emit(const uint32_t* __restrict__ order, const uint8_t* __restrict__ text, const uint32_t* __restrict__ starts,
               const uint32_t* __restrict__ lens, unsigned long long n, uint8_t* __restrict__ dict,
               unsigned long long* __restrict__ entry_off, long long* __restrict__ codes) {
  for (unsigned long long j = thread_index(); j < n; j += grid_threads()) {
    const uint32_t i = order[j];
    const unsigned long long a = entry_off[j] + 1;  // behind the origin byte
    const uint8_t* s = text + starts[i];
    const uint32_t L = lens[i];
    for (uint32_t k = 0; k <= L; ++k) dict[a + k] = s[k];  // the NUL too
    entry_off[j] = a;
    codes[i] = (long long)j;
    if (j == 0) {
      dict[0] = 0;
      entry_off[n] += 1;
    }
  }
}

unsigned grid_for(const Ctx* ctx, unsigned long long threads) {
  const unsigned long long want = (threads + NM_THREADS - 1) / NM_THREADS;
  const unsigned long long cap = (unsigned long long)ctx->sm_count * 16;
  return (unsigned)std::max<unsigned long long>(1, std::min(want, cap));
}

int check_opts(Ctx* ctx, const zdwb_number_opts* o, bool format, const char* who) {
  if (o->kind != ZDWB_NUM_DATETIME && o->kind != ZDWB_NUM_DECIMAL) {
    ctx->err = std::string(who) + ": kind " + std::to_string(o->kind) + " is neither ZDWB_NUM_DATETIME nor ZDWB_NUM_DECIMAL";
    return ZDWB_ERR_BAD_ARG;
  }
  // DATETIME parse ignores digits
  const int hi = o->kind == ZDWB_NUM_DECIMAL ? 18 : 6;
  if ((o->kind == ZDWB_NUM_DECIMAL || format) && (o->digits < 0 || o->digits > hi)) {
    ctx->err = std::string(who) + ": digits " + std::to_string(o->digits) + " is outside 0.." + std::to_string(hi);
    return ZDWB_ERR_BAD_ARG;
  }
  return ZDWB_OK;
}

}  // namespace

int parse_numbers_impl(Ctx* ctx, const zdwb_code_part* d, const zdwb_number_opts* o, zdwb_parse_out* out) {
  memset(out, 0, sizeof(*out));
  const char* who = "parse_numbers";
  ZDWB_TRY(check_dict(ctx, d, who));
  ZDWB_TRY(check_opts(ctx, o, false, who));
  if (o->null_text_len && !o->null_text) {
    ctx->err = "parse_numbers: NULL null_text with a length";
    return ZDWB_ERR_BAD_ARG;
  }
  ZDWB_TRY(call_begin(ctx));
  const unsigned long long E = d->entries;
  DevBuf d_null, d_bad;
  ZDWB_TRY(upload_host(ctx, d_null, o->null_text, o->null_text_len, who));
  ZDWB_TRY(d_bad.alloc(ctx, 8));
  ZDWB_CUDA_TRY(ctx, cudaMemsetAsync(d_bad.p, 0xff, 8, ctx->stream));
  long long* values;
  uint8_t* ok;
  {
    DevBuf vb, ob;
    ZDWB_TRY(vb.alloc(ctx, (E + 1) * 8));
    ZDWB_TRY(ob.alloc(ctx, E + 1));
    ok = static_cast<uint8_t*>(ob.detach());
    values = static_cast<long long*>(vb.detach());
  }
  ZDWB_TRY(launch(ctx, "k_num_parse", k_num_parse, grid_for(ctx, E + 1), NM_THREADS, 0, d->dict, d->entry_off, E, d->dict_bytes,
                  (const uint8_t*)d_null.as<uint8_t>(), (unsigned long long)o->null_text_len, (int)o->kind, (uint32_t)o->digits,
                  values, ok, d_bad.as<unsigned long long>()));
  unsigned long long bad;
  ZDWB_TRY(read_back(ctx, d_bad.p, &bad));
  if (bad != NM_NONE) {
    ctx->err = "parse_numbers: entry " + std::to_string(bad) + " has offsets that are not entry_off[e] < entry_off[e+1] <= dict_bytes";
    return ZDWB_ERR_BAD_ARG;
  }
  out->values = reinterpret_cast<const int64_t*>(values);
  out->ok = ok;
  out->n = E + 1;
  return ZDWB_OK;
}

int format_numbers_impl(Ctx* ctx, const int64_t* values, uint64_t n, const zdwb_number_opts* o, zdwb_merge_out* out) {
  memset(out, 0, sizeof(*out));
  const char* who = "format_numbers";
  ZDWB_TRY(check_opts(ctx, o, true, who));
  if (n && !values) {
    ctx->err = "format_numbers: n > 0 with NULL values";
    return ZDWB_ERR_BAD_ARG;
  }
  if (n >= (1ull << 32)) {  // every text takes 2 bytes at the least
    ctx->err = "format_numbers: " + std::to_string(n) + " values give texts of 2^32 bytes or more (not supported)";
    return ZDWB_ERR_UNSUPPORTED;
  }
  ZDWB_TRY(call_begin(ctx));
  cudaStream_t st = ctx->stream;
  unsigned long long* entry_off;
  {
    DevBuf eb;
    ZDWB_TRY(eb.alloc(ctx, (n + 1) * 8));
    entry_off = static_cast<unsigned long long*>(eb.detach());
  }
  if (n == 0) {
    ZDWB_CUDA_TRY(ctx, cudaMemsetAsync(entry_off, 0, 8, st));
    ZDWB_CUDA_TRY(ctx, cudaStreamSynchronize(st));
    out->entry_off = reinterpret_cast<const uint64_t*>(entry_off);
    return ZDWB_OK;
  }
  long long* codes;
  {
    DevBuf cb;
    ZDWB_TRY(cb.alloc(ctx, n * 8));
    codes = static_cast<long long*>(cb.detach());
  }
  const int kind = o->kind;
  const uint32_t digits = (uint32_t)o->digits;
  const long long* v = reinterpret_cast<const long long*>(values);
  const unsigned g = grid_for(ctx, n);

  // 1. checks and lengths, 2. lengths -> offsets; one round trip for the fault word and the total
  DevBuf d_meta, d_off;
  ZDWB_TRY(d_meta.alloc(ctx, sizeof(FormatMeta)));
  FormatMeta* meta = d_meta.as<FormatMeta>();
  ZDWB_CUDA_TRY(ctx, cudaMemsetAsync(meta, 0xff, 8, st));
  ZDWB_TRY(d_off.alloc(ctx, n * 8));
  unsigned long long* off = d_off.as<unsigned long long>();
  ZDWB_TRY(launch(ctx, "k_num_check", k_num_check, g, NM_THREADS, 0, v, n, kind, digits, off, meta));
  ZDWB_TRY(exclusive_scan_u64(ctx, reinterpret_cast<uint64_t*>(off), reinterpret_cast<uint64_t*>(off), n,
                              reinterpret_cast<uint64_t*>(&meta->total)));
  FormatMeta h;
  ZDWB_TRY(read_back(ctx, meta, &h));
  if (h.bad != NM_NONE) {
    const unsigned long long i = h.bad >> 2;
    const unsigned long long why = h.bad & 3;
    ctx->err = "format_numbers: value " + std::to_string(i) +
               (why == NM_ORDER ? " is not greater than the value before it (the values must be strictly increasing)"
                : why == NM_RANGE ? " is a DATETIME outside 0001-01-01 00:00:00 .. 9999-12-31 23:59:59.999999"
                                  : " is not a multiple of 10^" + std::to_string(6 - digits) + " microseconds (" +
                                        std::to_string(digits) + " fraction digits)");
    return ZDWB_ERR_BAD_ARG;
  }
  if (h.total >= (1ull << 32)) {
    ctx->err = "format_numbers: the texts take " + std::to_string(h.total) + " bytes with their terminators (2^32 and more are not supported)";
    return ZDWB_ERR_UNSUPPORTED;
  }

  // 3. the texts, 4. their bytewise order
  DevBuf d_text, d_starts, d_lens, d_order;
  ZDWB_TRY(d_text.alloc(ctx, h.total));
  ZDWB_TRY(d_starts.alloc(ctx, n * 4));
  ZDWB_TRY(d_lens.alloc(ctx, n * 4));
  ZDWB_TRY(d_order.alloc(ctx, n * 4));
  uint8_t* text = d_text.as<uint8_t>();
  ZDWB_TRY(launch(ctx, "k_num_write", k_num_write, g, NM_THREADS, 0, v, n, kind, digits, (const unsigned long long*)off, text,
                  d_starts.as<uint32_t>(), d_lens.as<uint32_t>()));
  const uint32_t max_len = kind == ZDWB_NUM_DATETIME ? 26u : 21u + digits;  // '-', 19 digits, '.' and the fraction at most
  ZDWB_TRY(sort_strings(ctx, text, d_starts.as<uint32_t>(), d_lens.as<uint32_t>(), (uint32_t)n, max_len, d_order.as<uint32_t>()));

  // 5. the dictionary in that order, its offsets and the codes
  uint8_t* dict;
  {
    DevBuf db;
    ZDWB_TRY(db.alloc(ctx, 1 + h.total));
    dict = static_cast<uint8_t*>(db.detach());
  }
  ZDWB_TRY(launch(ctx, "k_num_sorted_lens", k_num_sorted_lens, g, NM_THREADS, 0, (const uint32_t*)d_order.as<uint32_t>(),
                  (const uint32_t*)d_lens.as<uint32_t>(), n, entry_off));
  ZDWB_TRY(exclusive_scan_u64(ctx, reinterpret_cast<uint64_t*>(entry_off), reinterpret_cast<uint64_t*>(entry_off), n,
                              reinterpret_cast<uint64_t*>(entry_off + n)));
  ZDWB_TRY(launch(ctx, "k_num_emit", k_num_emit, g, NM_THREADS, 0, (const uint32_t*)d_order.as<uint32_t>(), (const uint8_t*)text,
                  (const uint32_t*)d_starts.as<uint32_t>(), (const uint32_t*)d_lens.as<uint32_t>(), n, dict, entry_off, codes));
  ZDWB_CUDA_TRY(ctx, cudaStreamSynchronize(st));
  out->codes = reinterpret_cast<const int64_t*>(codes);
  out->dict = dict;
  out->entry_off = reinterpret_cast<const uint64_t*>(entry_off);
  out->entries = n;
  out->dict_bytes = 1 + h.total;
  out->n = n;
  return ZDWB_OK;
}

}  // namespace zdwb
