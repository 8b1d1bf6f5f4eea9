// merge.cu -- zdwb_merge_codes: one sorted, dense dictionary for codes that point into many sorted dictionaries.
//
// Every input part is a dictionary whose entries are sorted and distinct (a block's dictionary, DESIGN 4.5) and codes
// into it.  The referenced entries of a part form a sorted run; the runs are merged pairwise, ceil(log2 P) levels, and
// a string found in both runs of a pair is kept once.  Kernels, in order (DESIGN 4.6):
//   k_merge_mark     one pass over all codes: range check, flag the referenced entries, count them
//   (scan)           flags -> the index of every referenced entry among all references ("refs")
//   k_merge_compact  refs in part order, with each ref's 16-byte prefix key and string; checks the entry's offsets
//   k_merge_runs     where every part's run starts
//   k_merge_check    every run strictly increasing
//   per level: k_merge_place (place in the merged pair, flag duplicates), (scan), k_merge_move (compact), k_merge_follow
//   k_merge_lengths, (scan), k_merge_emit  the output dictionary and its entry offsets
//   k_merge_remap    one pass over all codes: out = final index of the code's ref
// Nothing is read through an entry's offsets before they have been checked, so garbage input cannot fault the GPU.
#include "common.cuh"

namespace zdwb {

namespace {

constexpr int MG_THREADS = 256;

// a part as the kernels see it
struct MergePart {
  const uint8_t* dict;
  const uint64_t* entry_off;
  const int64_t* codes;
  uint64_t entries;
  uint64_t dict_bytes;
};

// device-side results of the call, read back by the host between stages
struct MergeMeta {
  uint32_t err;        // MG_ERR_* bits
  uint32_t bad_part;   // lowest part with an error
  unsigned long long refs;  // referenced entries
  uint32_t m[2];       // elements of the current / next level
  unsigned long long bytes;  // sum over output entries of (length + 1)
};
constexpr uint32_t MG_ERR_CODE = 1, MG_ERR_OFFSETS = 2, MG_ERR_ORDER = 4;

__device__ __forceinline__ void merge_fail(MergeMeta* meta, uint32_t bit, uint32_t part) {
  atomicOr(&meta->err, bit);
  atomicMin(&meta->bad_part, part);
}

// the last i with a[i] <= x (a ascending, a[0] <= x)
template <typename T>
__device__ __forceinline__ uint32_t last_le(const T* __restrict__ a, uint32_t n, unsigned long long x) {
  uint32_t lo = 0, hi = n;  // answer in [lo, hi)
  while (hi - lo > 1) {
    const uint32_t mid = (lo + hi) >> 1;
    if ((unsigned long long)a[mid] <= x) lo = mid;
    else hi = mid;
  }
  return lo;
}

__device__ __forceinline__ unsigned long long grid_threads() { return (unsigned long long)gridDim.x * blockDim.x; }
__device__ __forceinline__ unsigned long long thread_index() { return (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; }

// Every code: range check, and a flag on the entry it references.  The first thread to flag an entry counts it.
__global__ void __launch_bounds__(MG_THREADS)
    k_merge_mark(const MergePart* __restrict__ parts, const unsigned long long* __restrict__ code_base,
                 const unsigned long long* __restrict__ ent_base, uint32_t P, unsigned long long N, uint32_t* __restrict__ flags,
                 MergeMeta* meta) {
  uint32_t fresh = 0;
  for (unsigned long long j = thread_index(); j < N; j += grid_threads()) {
    const uint32_t p = last_le(code_base, P + 1, j);
    const long long c = parts[p].codes[j - code_base[p]];
    if (c < -1 || (c >= 0 && (unsigned long long)c >= parts[p].entries)) {
      merge_fail(meta, MG_ERR_CODE, p);
    } else if (c >= 0) {
      uint32_t* f = flags + ent_base[p] + (unsigned long long)c;
      if (*f == 0u && atomicExch(f, 1u) == 0u) ++fresh;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) fresh += __shfl_down_sync(0xffffffffu, fresh, o);
  if (lane_id() == 0 && fresh) atomicAdd(&meta->refs, (unsigned long long)fresh);
}

// Every referenced entry e (pos[e + 1] > pos[e]; pos = exclusive scan of the flags) becomes ref pos[e]: its offsets are
// checked, then its string and 16-byte prefix key are stored.  An entry with bad offsets gets an empty string.
__global__ void __launch_bounds__(MG_THREADS)
    k_merge_compact(const MergePart* __restrict__ parts, const unsigned long long* __restrict__ ent_base, uint32_t P,
                    unsigned long long E, const uint32_t* __restrict__ pos, ulonglong2* __restrict__ keys, Str* __restrict__ strs,
                    MergeMeta* meta) {
  for (unsigned long long e = thread_index(); e < E; e += grid_threads()) {
    const uint32_t r = pos[e];
    if (pos[e + 1] == r) continue;
    const uint32_t p = last_le(ent_base, P + 1, e);
    const MergePart& pt = parts[p];
    const unsigned long long local = e - ent_base[p];
    const unsigned long long a = pt.entry_off[local], b = pt.entry_off[local + 1];
    Str s{nullptr, 0ull};
    ulonglong2 k = make_ulonglong2(0ull, 0ull);
    if (a < b && b <= pt.dict_bytes) {
      s.p = pt.dict + a;
      s.len = b - a - 1;
      k = make_ulonglong2(key8(s.p, s.len, 0), key8(s.p, s.len, 8));
    } else {
      merge_fail(meta, MG_ERR_OFFSETS, p);
    }
    keys[r] = k;
    strs[r] = s;
  }
}

// run_off[p] = the first ref of part p (run_off[P] = R); the level-0 element count
__global__ void k_merge_runs(const unsigned long long* __restrict__ ent_base, uint32_t P, const uint32_t* __restrict__ pos,
                             uint32_t* __restrict__ run_off, MergeMeta* meta) {
  const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p > P) return;
  run_off[p] = pos[ent_base[p]];
  if (p == P) meta->m[0] = pos[ent_base[P]];
}

// Each ref is greater than the ref before it in its part.
__global__ void __launch_bounds__(MG_THREADS)
    k_merge_check(const ulonglong2* __restrict__ keys, const Str* __restrict__ strs, const uint32_t* __restrict__ run_off,
                  uint32_t P, uint32_t R, MergeMeta* meta) {
  if (meta->err) return;  // (offsets failed: the run is not read)
  for (unsigned long long r = thread_index() + 1; r < R; r += grid_threads()) {
    const uint32_t q = last_le(run_off, P + 1, r);
    if (run_off[q] == r) continue;  // first of its run
    if (str_cmp(keys[r - 1], strs[r - 1], keys[r], strs[r]) >= 0) merge_fail(meta, MG_ERR_ORDER, q);
  }
}

// One merge level, step 1: the place of every element in its merged pair of runs.  An element of a left run moves up
// by the elements of the right run below it; an element of a right run by the elements of the left run at or below it,
// and is a duplicate when the largest of those equals it.  keep[place] = 0 for duplicates and for k >= M.
__global__ void __launch_bounds__(MG_THREADS)
    k_merge_place(const ulonglong2* __restrict__ keys, const Str* __restrict__ strs, const uint32_t* __restrict__ run_off,
                  uint32_t nr, uint32_t R, const uint32_t* __restrict__ m_cur, uint32_t* __restrict__ place,
                  uint32_t* __restrict__ keep) {
  const uint32_t M = *m_cur;
  for (unsigned long long t = thread_index(); t < R; t += grid_threads()) {
    const uint32_t k = (uint32_t)t;
    if (k >= M) {
      keep[k] = 0u;
      continue;
    }
    const uint32_t q = last_le(run_off, nr + 1, k);
    const uint32_t sib = q ^ 1u;
    if (sib >= nr) {  // an odd run at the end passes through
      place[k] = k;
      keep[k] = 1u;
      continue;
    }
    const bool left = (q & 1u) == 0u;
    uint32_t lo = run_off[sib], hi = run_off[sib + 1];
    const uint32_t s0 = lo;
    const ulonglong2 kk = keys[k];
    const Str ss = strs[k];
    bool dup = false;
    // left: count of sibling elements < x; right: count of sibling elements <= x
    while (lo < hi) {
      const uint32_t mid = (lo + hi) >> 1;
      const int c = str_cmp(keys[mid], strs[mid], kk, ss);
      if (c < 0 || (!left && c == 0)) {
        lo = mid + 1;
        if (c == 0) dup = true;
      } else {
        hi = mid;
      }
    }
    const uint32_t pl = k + (lo - s0) - (left ? 0u : (run_off[q] - run_off[sib]));
    // (a right element's own index counts the left run's elements already; remove them, add those at or below it)
    place[k] = pl;
    keep[pl] = dup ? 0u : 1u;
  }
}

// Step 2 (after the scan of keep): the kept elements move to their compacted index; every element (duplicates too)
// records that index in new_idx; the runs of the next level are the pairs of this one.
__global__ void __launch_bounds__(MG_THREADS)
    k_merge_move(const ulonglong2* __restrict__ keys, const Str* __restrict__ strs, const uint32_t* __restrict__ run_off,
                 uint32_t nr, uint32_t R, const uint32_t* __restrict__ m_cur, const uint32_t* __restrict__ m_next,
                 const uint32_t* __restrict__ place, const uint32_t* __restrict__ excl, ulonglong2* __restrict__ keys_out,
                 Str* __restrict__ strs_out, uint32_t* __restrict__ new_idx, uint32_t* __restrict__ run_out) {
  const uint32_t M = *m_cur, total = *m_next;
  const uint32_t nr_next = (nr + 1) / 2;
  for (unsigned long long i = thread_index(); i <= nr_next; i += grid_threads()) {
    const uint32_t o = run_off[min(2u * (uint32_t)i, nr)];
    run_out[i] = o < R ? excl[o] : total;
  }
  for (unsigned long long t = thread_index(); t < M; t += grid_threads()) {
    const uint32_t k = (uint32_t)t, pl = place[k];
    const uint32_t nx = pl + 1 < R ? excl[pl + 1] : total;
    const bool kept = nx != excl[pl];
    const uint32_t n = kept ? excl[pl] : excl[pl] - 1u;  // a duplicate sits right behind its equal
    if (kept) {
      keys_out[n] = keys[k];
      strs_out[n] = strs[k];
    }
    new_idx[k] = n;
  }
}

// Step 3: every ref follows its element (level 0: the element is the ref itself; no new_idx: cur = identity).
__global__ void __launch_bounds__(MG_THREADS)
    k_merge_follow(uint32_t R, bool first, const uint32_t* __restrict__ new_idx, uint32_t* __restrict__ cur) {
  for (unsigned long long t = thread_index(); t < R; t += grid_threads())
    cur[t] = new_idx ? new_idx[first ? (uint32_t)t : cur[t]] : (uint32_t)t;
}

// entry lengths + 1 (the NUL), 0 past the last entry
__global__ void __launch_bounds__(MG_THREADS)
    k_merge_lengths(const Str* __restrict__ strs, uint32_t R, const uint32_t* __restrict__ m_cur,
                    unsigned long long* __restrict__ lens) {
  const uint32_t D = *m_cur;
  for (unsigned long long t = thread_index(); t < R; t += grid_threads()) lens[t] = t < D ? strs[t].len + 1ull : 0ull;
}

// One warp per entry: its bytes and its NUL at 1 + start[k]; the origin NUL and the closing offset.
__global__ void __launch_bounds__(MG_THREADS)
    k_merge_emit(const Str* __restrict__ strs, uint32_t D, const unsigned long long* __restrict__ start,
                 unsigned long long total, uint8_t* __restrict__ dict, unsigned long long* __restrict__ entry_off) {
  const unsigned long long w0 = thread_index() >> 5, nw = grid_threads() >> 5;
  const uint32_t lane = lane_id();
  if (thread_index() == 0) {
    dict[0] = 0;
    entry_off[D] = 1ull + total;
  }
  for (unsigned long long k = w0; k < D; k += nw) {
    const Str s = strs[k];
    const unsigned long long o = 1ull + start[k];
    if (lane == 0) {
      entry_off[k] = o;
      dict[o + s.len] = 0;
    }
    uint8_t* d = dict + o;
    unsigned long long i = lane;
    // 16-byte chunks where source and destination share their alignment, bytes elsewhere
    if (s.len >= 64 && (((uintptr_t)s.p ^ (uintptr_t)d) & 15u) == 0u) {
      const unsigned long long head = (16u - ((uintptr_t)d & 15u)) & 15u;
      for (i = lane; i < head; i += 32) d[i] = __ldg(s.p + i);
      const unsigned long long nch = (s.len - head) / 16;
      for (unsigned long long c = lane; c < nch; c += 32)
        reinterpret_cast<uint4*>(d + head)[c] = __ldg(reinterpret_cast<const uint4*>(s.p + head) + c);
      i = head + nch * 16 + lane;
    }
    for (; i < s.len; i += 32) d[i] = __ldg(s.p + i);
  }
}

// out[j] = the final index of the ref of code j (-1 stays -1)
__global__ void __launch_bounds__(MG_THREADS)
    k_merge_remap(const MergePart* __restrict__ parts, const unsigned long long* __restrict__ code_base,
                  const unsigned long long* __restrict__ ent_base, uint32_t P, unsigned long long N,
                  const uint32_t* __restrict__ pos, const uint32_t* __restrict__ cur, long long* __restrict__ out) {
  for (unsigned long long j = thread_index(); j < N; j += grid_threads()) {
    const uint32_t p = last_le(code_base, P + 1, j);
    const long long c = parts[p].codes[j - code_base[p]];
    out[j] = c < 0 ? -1ll : (long long)cur[pos[ent_base[p] + (unsigned long long)c]];
  }
}

unsigned grid_for(const Ctx* ctx, unsigned long long n) {
  const unsigned long long want = (n + MG_THREADS - 1) / MG_THREADS;
  const unsigned long long cap = (unsigned long long)ctx->sm_count * 8;
  return (unsigned)std::max<unsigned long long>(1, std::min(want, cap));
}

template <typename T>
int merge_upload(Ctx* ctx, DevBuf& d, const std::vector<T>& v) {
  ZDWB_TRY(d.alloc(ctx, v.size() * sizeof(T) + 16));
  const size_t n = v.size() * sizeof(T);
  void* pinned = stage_take(ctx, n);
  if (!pinned) {
    ctx->err = "merge_codes: pinned staging allocation failed";
    return ZDWB_ERR_OOM;
  }
  memcpy(pinned, v.data(), n);
  ZDWB_CUDA_TRY(ctx, cudaMemcpyAsync(d.p, pinned, n, cudaMemcpyHostToDevice, ctx->stream));
  return ZDWB_OK;
}

int read_meta(Ctx* ctx, const DevBuf& meta, MergeMeta* h) {
  ZDWB_CUDA_TRY(ctx, cudaMemcpyAsync(ctx->meta_host, meta.p, sizeof(MergeMeta), cudaMemcpyDeviceToHost, ctx->stream));
  ZDWB_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  memcpy(h, ctx->meta_host, sizeof(MergeMeta));
  return ZDWB_OK;
}

}  // namespace

int merge_codes_impl(Ctx* ctx, const zdwb_code_part* parts, uint32_t P, unsigned long long max_refs, zdwb_merge_out* out) {
  memset(out, 0, sizeof(*out));
  ZDWB_TRY(call_begin(ctx));
  cudaStream_t st = ctx->stream;
  if (P > 0 && !parts) {
    ctx->err = "merge_codes: parts is NULL";
    return ZDWB_ERR_BAD_ARG;
  }
  std::vector<MergePart> hp(P);
  std::vector<unsigned long long> code_base(P + 1, 0), ent_base(P + 1, 0);
  for (uint32_t p = 0; p < P; ++p) {
    const zdwb_code_part& q = parts[p];
    if (q.n > 0 && !q.codes) {
      ctx->err = "merge_codes: part " + std::to_string(p) + " has codes but a NULL codes pointer";
      return ZDWB_ERR_BAD_ARG;
    }
    if (q.entries > 0 && (!q.dict || !q.entry_off)) {
      ctx->err = "merge_codes: part " + std::to_string(p) + " has entries but a NULL dict or entry_off";
      return ZDWB_ERR_BAD_ARG;
    }
    hp[p] = MergePart{q.dict, q.entry_off, q.codes, q.entries, q.dict_bytes};
    code_base[p + 1] = code_base[p] + q.n;
    ent_base[p + 1] = ent_base[p] + q.entries;
  }
  const unsigned long long N = code_base[P], E = ent_base[P];
  out->n = N;

  DevBuf d_parts, d_code_base, d_ent_base, d_meta, d_pos;
  ZDWB_TRY(merge_upload(ctx, d_parts, hp));
  ZDWB_TRY(merge_upload(ctx, d_code_base, code_base));
  ZDWB_TRY(merge_upload(ctx, d_ent_base, ent_base));
  ZDWB_TRY(d_meta.alloc(ctx, sizeof(MergeMeta)));
  ZDWB_CUDA_TRY(ctx, cudaMemsetAsync(d_meta.p, 0, sizeof(MergeMeta), st));
  ZDWB_CUDA_TRY(ctx, cudaMemsetAsync(&d_meta.as<MergeMeta>()->bad_part, 0xff, 4, st));
  MergeMeta* meta = d_meta.as<MergeMeta>();
  const MergePart* dp = d_parts.as<MergePart>();
  const unsigned long long* dcb = d_code_base.as<unsigned long long>();
  const unsigned long long* deb = d_ent_base.as<unsigned long long>();

  // ---- mark and count the referenced entries; pos = their index among all refs (pos[E] = R)
  ZDWB_TRY(d_pos.alloc(ctx, (E + 1) * 4));
  uint32_t* pos = d_pos.as<uint32_t>();
  ZDWB_CUDA_TRY(ctx, cudaMemsetAsync(pos, 0, (E + 1) * 4, st));
  if (N) ZDWB_TRY(launch(ctx, "k_merge_mark", k_merge_mark, grid_for(ctx, N), MG_THREADS, 0, dp, dcb, deb, P, N, pos, meta));
  MergeMeta h;
  ZDWB_TRY(read_meta(ctx, d_meta, &h));
  if (h.err) {
    ctx->err = "merge_codes: part " + std::to_string(h.bad_part) + " has a code < -1 or >= its number of entries";
    return ZDWB_ERR_BAD_ARG;
  }
  if (h.refs > max_refs) {
    ctx->err = "merge_codes: " + std::to_string(h.refs) + " referenced entries (at most " + std::to_string(max_refs) +
               " are supported)";
    return ZDWB_ERR_UNSUPPORTED;
  }
  const uint32_t R = (uint32_t)h.refs;
  if (E) ZDWB_TRY(exclusive_scan_u32(ctx, pos, pos, E, pos + E));

  // ---- the refs in part order, each part a run; check offsets and order
  DevBuf keyA, keyB, strA, strB, runA, runB, place, keep, new_idx, cur;
  const size_t Rz = std::max<uint32_t>(R, 1);
  ZDWB_TRY(keyA.alloc(ctx, Rz * sizeof(ulonglong2)));
  ZDWB_TRY(strA.alloc(ctx, Rz * sizeof(Str)));
  ZDWB_TRY(runA.alloc(ctx, ((size_t)P + 1) * 4));
  if (R) {
    ZDWB_TRY(launch(ctx, "k_merge_compact", k_merge_compact, grid_for(ctx, E), MG_THREADS, 0, dp, deb, P, E, (const uint32_t*)pos,
                    keyA.as<ulonglong2>(), strA.as<Str>(), meta));
  }
  ZDWB_TRY(launch(ctx, "k_merge_runs", k_merge_runs, (P + 1 + 255) / 256, 256, 0, deb, P, (const uint32_t*)pos, runA.as<uint32_t>(),
                  meta));
  if (R > 1) {
    ZDWB_TRY(launch(ctx, "k_merge_check", k_merge_check, grid_for(ctx, R), MG_THREADS, 0, (const ulonglong2*)keyA.as<ulonglong2>(),
                    (const Str*)strA.as<Str>(), (const uint32_t*)runA.as<uint32_t>(), P, R, meta));
  }
  ZDWB_TRY(read_meta(ctx, d_meta, &h));
  if (h.err) {
    ctx->err = "merge_codes: part " + std::to_string(h.bad_part) +
               ((h.err & MG_ERR_OFFSETS) ? " references an entry whose offsets are not entry_off[e] < entry_off[e+1] <= dict_bytes"
                                         : " references entries that are not strictly increasing bytewise");
    return ZDWB_ERR_BAD_ARG;
  }

  // ---- merge levels: runs of the pairs of the level before; m[lv & 1] holds the level's element count
  uint32_t nr = P;
  int lv = 0;
  if (R && P > 1) {
    ZDWB_TRY(keyB.alloc(ctx, Rz * sizeof(ulonglong2)));
    ZDWB_TRY(strB.alloc(ctx, Rz * sizeof(Str)));
    ZDWB_TRY(runB.alloc(ctx, ((size_t)P + 1) * 4));
    ZDWB_TRY(place.alloc(ctx, Rz * 4));
    ZDWB_TRY(keep.alloc(ctx, Rz * 4));
    ZDWB_TRY(new_idx.alloc(ctx, Rz * 4));
    ZDWB_TRY(cur.alloc(ctx, Rz * 4));
    DevBuf* K[2] = {&keyA, &keyB};
    DevBuf* S[2] = {&strA, &strB};
    DevBuf* RO[2] = {&runA, &runB};
    const unsigned g = grid_for(ctx, R);
    for (; nr > 1; ++lv) {
      const int a = lv & 1, b = a ^ 1;
      const uint32_t* m_cur = &meta->m[a];
      uint32_t* m_next = &meta->m[b];
      ZDWB_TRY(launch(ctx, "k_merge_place", k_merge_place, g, MG_THREADS, 0, (const ulonglong2*)K[a]->as<ulonglong2>(),
                      (const Str*)S[a]->as<Str>(), (const uint32_t*)RO[a]->as<uint32_t>(), nr, R, m_cur, place.as<uint32_t>(),
                      keep.as<uint32_t>()));
      ZDWB_TRY(exclusive_scan_u32(ctx, keep.as<uint32_t>(), keep.as<uint32_t>(), R, m_next));
      ZDWB_TRY(launch(ctx, "k_merge_move", k_merge_move, g, MG_THREADS, 0, (const ulonglong2*)K[a]->as<ulonglong2>(),
                      (const Str*)S[a]->as<Str>(), (const uint32_t*)RO[a]->as<uint32_t>(), nr, R, m_cur, (const uint32_t*)m_next,
                      (const uint32_t*)place.as<uint32_t>(), (const uint32_t*)keep.as<uint32_t>(), K[b]->as<ulonglong2>(),
                      S[b]->as<Str>(), new_idx.as<uint32_t>(), RO[b]->as<uint32_t>()));
      ZDWB_TRY(launch(ctx, "k_merge_follow", k_merge_follow, g, MG_THREADS, 0, R, lv == 0, (const uint32_t*)new_idx.as<uint32_t>(),
                      cur.as<uint32_t>()));
      nr = (nr + 1) / 2;
    }
  }
  const int fin = lv & 1;
  const Str* strs = (fin ? strB : strA).as<Str>();

  // ---- emit: entry lengths -> their starts -> the dictionary and its offsets
  DevBuf lens;
  ZDWB_TRY(lens.alloc(ctx, Rz * 8));
  if (R) {
    ZDWB_TRY(launch(ctx, "k_merge_lengths", k_merge_lengths, grid_for(ctx, R), MG_THREADS, 0, strs, R,
                    (const uint32_t*)&meta->m[fin], lens.as<unsigned long long>()));
    ZDWB_TRY(exclusive_scan_u64(ctx, lens.as<uint64_t>(), lens.as<uint64_t>(), R, reinterpret_cast<uint64_t*>(&meta->bytes)));
  }
  ZDWB_TRY(read_meta(ctx, d_meta, &h));
  const uint32_t D = R ? h.m[fin] : 0;
  const unsigned long long dict_bytes = D ? 1ull + h.bytes : 0ull;
  uint8_t* dict = nullptr;
  unsigned long long* entry_off;
  {
    DevBuf eb;
    ZDWB_TRY(eb.alloc(ctx, ((size_t)D + 1) * 8));
    entry_off = static_cast<unsigned long long*>(eb.detach());
  }
  if (D) {
    DevBuf db;
    ZDWB_TRY(db.alloc(ctx, dict_bytes));
    dict = static_cast<uint8_t*>(db.detach());
    ZDWB_TRY(launch(ctx, "k_merge_emit", k_merge_emit, grid_for(ctx, (unsigned long long)D * 32), MG_THREADS, 0, strs, D,
                    (const unsigned long long*)lens.as<unsigned long long>(), h.bytes, dict, entry_off));
  } else {
    ZDWB_CUDA_TRY(ctx, cudaMemsetAsync(entry_off, 0, 8, st));
  }

  // ---- the codes
  long long* codes = nullptr;
  if (N) {
    DevBuf cb;
    ZDWB_TRY(cb.alloc(ctx, N * 8));
    codes = static_cast<long long*>(cb.detach());
    // with one run the refs are final as they are: cur = identity
    if (!(R && P > 1)) {
      ZDWB_TRY(cur.alloc(ctx, Rz * 4));
      ZDWB_TRY(launch(ctx, "k_merge_follow", k_merge_follow, grid_for(ctx, R), MG_THREADS, 0, R, true, (const uint32_t*)nullptr,
                      cur.as<uint32_t>()));
    }
    ZDWB_TRY(launch(ctx, "k_merge_remap", k_merge_remap, grid_for(ctx, N), MG_THREADS, 0, dp, dcb, deb, P, N, (const uint32_t*)pos,
                    (const uint32_t*)cur.as<uint32_t>(), codes));
  }
  ZDWB_CUDA_TRY(ctx, cudaStreamSynchronize(st));
  out->codes = reinterpret_cast<const int64_t*>(codes);
  out->dict = dict;
  out->entry_off = reinterpret_cast<const uint64_t*>(entry_off);
  out->entries = D;
  out->dict_bytes = dict_bytes;
  return ZDWB_OK;
}

}  // namespace zdwb
