// ctx.cu -- C ABI entry points of libzdw_b200 (see include/zdw_b200.h).
#include <errno.h>
#include <unistd.h>

#include <map>
#include <new>

#include "common.cuh"

struct zdwb_ctx : zdwb::Ctx {
  long long merge_max_refs = 0xffffffffll;  // zdwb_merge_codes: most referenced entries of a call (tests lower it)
  void* render_dev = nullptr;  // zdwb_render_columns' output (own allocation: it outlives the arena resets of later calls)
  size_t render_dev_cap = 0;
};

namespace zdwb {
int encode_block_impl(Ctx* ctx, const zdwb_schema* schema, const void* tsv, size_t n, const zdwb_encode_opts* opts,
                      zdwb_block_out* out);
int decode_block_impl(Ctx* ctx, const zdwb_schema* schema, const void* zdw, size_t avail, const zdwb_decode_opts* opts,
                      zdwb_rows_out* out);
int decode_columns_impl(Ctx* ctx, const zdwb_schema* schema, const void* zdw, size_t avail, const zdwb_columns_opts* opts,
                        zdwb_columns_out* out);
int merge_codes_impl(Ctx* ctx, const zdwb_code_part* parts, uint32_t n_parts, unsigned long long max_refs, zdwb_merge_out* out);
int render_columns_impl(Ctx* ctx, const zdwb_schema* schema, const zdwb_code_part* cols, void** buf, size_t* cap,
                        zdwb_render_out* out);
int match_like_impl(Ctx* ctx, const zdwb_code_part* dict, const zdwb_like_opts* opts, zdwb_match_out* out);
int find_strings_impl(Ctx* ctx, const zdwb_code_part* dict, const zdwb_strings* queries, zdwb_find_out* out);
int parse_numbers_impl(Ctx* ctx, const zdwb_code_part* dict, const zdwb_number_opts* opts, zdwb_parse_out* out);
int format_numbers_impl(Ctx* ctx, const int64_t* values, uint64_t n, const zdwb_number_opts* opts, zdwb_merge_out* out);
}  // namespace zdwb

using zdwb::Ctx;

extern "C" {

int zdwb_abi_version(void) { return ZDWB_ABI_VERSION; }

int zdwb_device_count(void) {
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess) {
    (void)cudaGetLastError();
    return 0;
  }
  return count;
}

int zdwb_ctx_create(int device, size_t workspace_hint, zdwb_ctx** out) {
  if (!out) return ZDWB_ERR_BAD_ARG;
  *out = nullptr;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0) {
    (void)cudaGetLastError();
    return ZDWB_ERR_NO_DEVICE;  // no CPU fallback
  }
  if (device < 0 || device >= count) return ZDWB_ERR_BAD_ARG;
  if (cudaSetDevice(device) != cudaSuccess) return ZDWB_ERR_NO_DEVICE;
  zdwb_ctx* c = new (std::nothrow) zdwb_ctx();
  if (!c) return ZDWB_ERR_OOM;
  c->device = device;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) c->sm_count = prop.multiProcessorCount;
  if (cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking) != cudaSuccess) {
    delete c;
    return ZDWB_ERR_CUDA;
  }
  c->stream = c->own_stream;
  // (mapped: kernels store small results straight into it, decode.cu k_readback)
  if (cudaHostAlloc(&c->meta_host, 4096, cudaHostAllocMapped | cudaHostAllocPortable) != cudaSuccess) {
    cudaStreamDestroy(c->own_stream);
    delete c;
    return ZDWB_ERR_OOM;
  }
  if (workspace_hint) {  // size the arena up front
    void* p = arena_alloc(c, workspace_hint);
    if (p) arena_release(c, p, workspace_hint);
  }
  *out = c;
  return ZDWB_OK;
}

void zdwb_ctx_destroy(zdwb_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  arena_destroy(c);
  out_host_release(c);
  if (c->out_host2) cudaFreeHost(c->out_host2);
  if (c->meta_host) cudaFreeHost(c->meta_host);
  if (c->stage_host) cudaFreeHost(c->stage_host);
  zdwb::ring_destroy(c);
  if (c->fd_dev) cudaFree(c->fd_dev);
  if (c->render_dev) cudaFree(c->render_dev);
  if (c->own_stream) cudaStreamDestroy(c->own_stream);
  delete c;
}

// ---- file descriptor <-> device, through the pinned ring ----------------------------------------------------------
int zdwb_fd_to_device(zdwb_ctx* c, int fd, long long offset, size_t len, const void** dev) {
  if (!c || !dev || fd < 0) return ZDWB_ERR_BAD_ARG;
  *dev = nullptr;
  c->err.clear();
  if (cudaSetDevice(c->device) != cudaSuccess) return ZDWB_ERR_NO_DEVICE;
  if (c->fd_dev_cap < len + 64) {
    ZDWB_CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    if (c->fd_dev) cudaFree(c->fd_dev);
    c->fd_dev = nullptr;
    c->fd_dev_cap = 0;
    const size_t cap = len + len / 8 + 64;  // headroom: the windows of a file vary a little
    ZDWB_CUDA_TRY(c, cudaMalloc(&c->fd_dev, cap));
    c->fd_dev_cap = cap;
  }
  int rc;
  try {
  rc = zdwb::ring_h2d(c, c->fd_dev, len, [fd, offset, c](void* dst, size_t off, size_t n) {
    size_t got = 0;
    while (got < n) {
      const ssize_t r = offset >= 0 ? pread(fd, static_cast<char*>(dst) + got, n - got, (off_t)((size_t)offset + off + got))
                                    : read(fd, static_cast<char*>(dst) + got, n - got);
      if (r < 0 && errno == EINTR) continue;
      if (r <= 0) {
        c->err = r == 0 ? "fd_to_device: the input ended early" : std::string("fd_to_device: read failed: ") + strerror(errno);
        return false;
      }
      got += (size_t)r;
    }
    return true;
  });
  } catch (...) {  // (nothing of the host side's C++ may leave through the C ABI)
    c->err = "zdwb_fd_to_device: out of host memory";
    return ZDWB_ERR_OOM;
  }
  if (rc != ZDWB_OK) return rc;
  *dev = c->fd_dev;
  return ZDWB_OK;
}

int zdwb_device_to_fd(zdwb_ctx* c, const void* dev, size_t len, int fd, long long offset) {
  if (!c || (!dev && len) || fd < 0) return ZDWB_ERR_BAD_ARG;
  c->err.clear();
  if (cudaSetDevice(c->device) != cudaSuccess) return ZDWB_ERR_NO_DEVICE;
  try {
  return zdwb::ring_d2h(c, dev, len, [fd, offset, c](const uint8_t* src, size_t off, size_t n) {
    size_t put = 0;
    while (put < n) {
      const ssize_t w = offset >= 0 ? pwrite(fd, src + put, n - put, (off_t)((size_t)offset + off + put)) : write(fd, src + put, n - put);
      if (w < 0 && errno == EINTR) continue;
      if (w <= 0) {
        c->err = std::string("device_to_fd: write failed: ") + strerror(errno);
        return false;
      }
      put += (size_t)w;
    }
    return true;
  });
  } catch (...) {
    c->err = "zdwb_device_to_fd: out of host memory";
    return ZDWB_ERR_OOM;
  }
}

const char* zdwb_last_error(const zdwb_ctx* c) { return c ? c->err.c_str() : "null context"; }

int zdwb_ctx_set_stream(zdwb_ctx* c, void* cuda_stream) {
  if (!c) return ZDWB_ERR_BAD_ARG;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  c->stream = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : c->own_stream;
  return ZDWB_OK;
}

int zdwb_ctx_set_tuning(zdwb_ctx* c, const char* name, long long value) {
  if (!c || !name) return ZDWB_ERR_BAD_ARG;
  if (!strcmp(name, "small_sort_max")) c->small_sort_max = value;
  else if (!strcmp(name, "sort_radix_items")) c->sort_radix_items = value;
  else if (!strcmp(name, "ht_initial_log2")) c->ht_initial_log2 = value;
  else if (!strcmp(name, "dec_tile_bytes")) c->dec_tile_bytes = value;
  else if (!strcmp(name, "copy_gate")) c->copy_gate = value;
  else if (!strcmp(name, "dec_delta")) c->dec_delta = value;
  else if (!strcmp(name, "dec_strip_rows")) c->dec_strip_rows = value;
  else if (!strcmp(name, "dec_group_lanes")) c->dec_group_lanes = value;
  else if (!strcmp(name, "enc_delta")) {
    c->enc_delta = value;
    c->delta_bailed = false;
  } else if (!strcmp(name, "enc_p2_rows")) c->enc_p2_rows = value;
  else if (!strcmp(name, "enc_dtile")) c->enc_dtile = value;
  else if (!strcmp(name, "enc_census")) {
    c->enc_census = value;
    c->census_fell_back = false;
  }
  else if (!strcmp(name, "merge_max_refs")) c->merge_max_refs = value < 0 ? 0 : value > 0xffffffffll ? 0xffffffffll : value;
  else if (!strcmp(name, "kernel_timing")) c->timing = value != 0;
  else return ZDWB_ERR_BAD_ARG;
  return ZDWB_OK;
}

unsigned long long zdwb_ctx_kernel_launches(const zdwb_ctx* c) { return c ? c->launches : 0ull; }

size_t zdwb_ctx_kernel_times(zdwb_ctx* c, char* buf, size_t cap) {
  if (!c) return 0;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  try {
    std::map<std::string, std::pair<unsigned long long, double>> agg;
    for (auto& t : c->timed) {
      float ms = 0.f;
      if (cudaEventElapsedTime(&ms, t.e0, t.e1) == cudaSuccess) {
        auto& a = agg[t.name];
        a.first += 1;
        a.second += ms;
      }
      cudaEventDestroy(t.e0);
      cudaEventDestroy(t.e1);
    }
    c->timed.clear();
    (void)cudaGetLastError();
    std::string out;
    for (auto& kv : agg) {
      char line[256];
      snprintf(line, sizeof(line), "%s\t%llu\t%.6f\n", kv.first.c_str(), kv.second.first, kv.second.second);
      out += line;
    }
    if (buf && cap) {
      const size_t k = out.size() < cap - 1 ? out.size() : cap - 1;
      memcpy(buf, out.data(), k);
      buf[k] = 0;
    }
    return out.size();
  } catch (...) {  // out of host memory while formatting: report nothing rather than throw through the C ABI
    if (buf && cap) buf[0] = 0;
    return 0;
  }
}

int zdwb_encode_block(zdwb_ctx* c, const zdwb_schema* schema, const void* tsv, size_t n, const zdwb_encode_opts* opts,
                      zdwb_block_out* out) {
  if (!c) return ZDWB_ERR_BAD_ARG;
  c->err.clear();
  if (!schema || !out || !opts || (!tsv && n)) {
    c->err = "zdwb_encode_block: null argument";
    return ZDWB_ERR_BAD_ARG;
  }
  if (cudaSetDevice(c->device) != cudaSuccess) {
    c->err = "cudaSetDevice failed";
    return ZDWB_ERR_NO_DEVICE;
  }
  // the implementation uses std::vector / std::string on the host side: nothing of that may leave through the C ABI
  try {
    return zdwb::encode_block_impl(c, schema, tsv, n, opts, out);
  } catch (const std::bad_alloc&) {
    c->err = "zdwb_encode_block: out of host memory";
    return ZDWB_ERR_OOM;
  } catch (...) {
    c->err = "zdwb_encode_block: unexpected C++ exception";
    return ZDWB_ERR_CUDA;
  }
}

int zdwb_decode_block(zdwb_ctx* c, const zdwb_schema* schema, const void* zdw, size_t avail, const zdwb_decode_opts* opts,
                      zdwb_rows_out* out) {
  if (!c) return ZDWB_ERR_BAD_ARG;
  c->err.clear();
  if (!schema || !out || !opts || !zdw) {
    c->err = "zdwb_decode_block: null argument";
    return ZDWB_ERR_BAD_ARG;
  }
  if (cudaSetDevice(c->device) != cudaSuccess) {
    c->err = "cudaSetDevice failed";
    return ZDWB_ERR_NO_DEVICE;
  }
  try {
    return zdwb::decode_block_impl(c, schema, zdw, avail, opts, out);
  } catch (const std::bad_alloc&) {
    c->err = "zdwb_decode_block: out of host memory";
    return ZDWB_ERR_OOM;
  } catch (...) {
    c->err = "zdwb_decode_block: unexpected C++ exception";
    return ZDWB_ERR_CUDA;
  }
}

int zdwb_decode_columns(zdwb_ctx* c, const zdwb_schema* schema, const void* zdw, size_t avail, const zdwb_columns_opts* opts,
                        zdwb_columns_out* out) {
  if (!c) return ZDWB_ERR_BAD_ARG;
  c->err.clear();
  if (!schema || !out || !opts || !zdw) {
    c->err = "zdwb_decode_columns: null argument";
    return ZDWB_ERR_BAD_ARG;
  }
  if (cudaSetDevice(c->device) != cudaSuccess) {
    c->err = "cudaSetDevice failed";
    return ZDWB_ERR_NO_DEVICE;
  }
  try {
    return zdwb::decode_columns_impl(c, schema, zdw, avail, opts, out);
  } catch (const std::bad_alloc&) {
    c->err = "zdwb_decode_columns: out of host memory";
    return ZDWB_ERR_OOM;
  } catch (...) {
    c->err = "zdwb_decode_columns: unexpected C++ exception";
    return ZDWB_ERR_CUDA;
  }
}

int zdwb_merge_codes(zdwb_ctx* c, const zdwb_code_part* parts, uint32_t n_parts, zdwb_merge_out* out) {
  if (!c) return ZDWB_ERR_BAD_ARG;
  c->err.clear();
  if (!out) {
    c->err = "zdwb_merge_codes: null argument";
    return ZDWB_ERR_BAD_ARG;
  }
  if (cudaSetDevice(c->device) != cudaSuccess) {
    c->err = "cudaSetDevice failed";
    return ZDWB_ERR_NO_DEVICE;
  }
  try {
    return zdwb::merge_codes_impl(c, parts, n_parts, (unsigned long long)c->merge_max_refs, out);
  } catch (const std::bad_alloc&) {
    c->err = "zdwb_merge_codes: out of host memory";
    return ZDWB_ERR_OOM;
  } catch (...) {
    c->err = "zdwb_merge_codes: unexpected C++ exception";
    return ZDWB_ERR_CUDA;
  }
}

int zdwb_render_columns(zdwb_ctx* c, const zdwb_schema* schema, const zdwb_code_part* cols, zdwb_render_out* out) {
  if (!c) return ZDWB_ERR_BAD_ARG;
  c->err.clear();
  if (!schema || !cols || !out) {
    c->err = "zdwb_render_columns: null argument";
    return ZDWB_ERR_BAD_ARG;
  }
  if (cudaSetDevice(c->device) != cudaSuccess) {
    c->err = "cudaSetDevice failed";
    return ZDWB_ERR_NO_DEVICE;
  }
  try {
    return zdwb::render_columns_impl(c, schema, cols, &c->render_dev, &c->render_dev_cap, out);
  } catch (const std::bad_alloc&) {
    c->err = "zdwb_render_columns: out of host memory";
    return ZDWB_ERR_OOM;
  } catch (...) {
    c->err = "zdwb_render_columns: unexpected C++ exception";
    return ZDWB_ERR_CUDA;
  }
}

int zdwb_match_like(zdwb_ctx* c, const zdwb_code_part* dict, const zdwb_like_opts* opts, zdwb_match_out* out) {
  if (!c) return ZDWB_ERR_BAD_ARG;
  c->err.clear();
  if (!opts || !out) {
    c->err = "zdwb_match_like: null argument";
    return ZDWB_ERR_BAD_ARG;
  }
  if (cudaSetDevice(c->device) != cudaSuccess) {
    c->err = "cudaSetDevice failed";
    return ZDWB_ERR_NO_DEVICE;
  }
  try {
    return zdwb::match_like_impl(c, dict, opts, out);
  } catch (const std::bad_alloc&) {
    c->err = "zdwb_match_like: out of host memory";
    return ZDWB_ERR_OOM;
  } catch (...) {
    c->err = "zdwb_match_like: unexpected C++ exception";
    return ZDWB_ERR_CUDA;
  }
}

int zdwb_find_strings(zdwb_ctx* c, const zdwb_code_part* dict, const zdwb_strings* queries, zdwb_find_out* out) {
  if (!c) return ZDWB_ERR_BAD_ARG;
  c->err.clear();
  if (!queries || !out) {
    c->err = "zdwb_find_strings: null argument";
    return ZDWB_ERR_BAD_ARG;
  }
  if (cudaSetDevice(c->device) != cudaSuccess) {
    c->err = "cudaSetDevice failed";
    return ZDWB_ERR_NO_DEVICE;
  }
  try {
    return zdwb::find_strings_impl(c, dict, queries, out);
  } catch (const std::bad_alloc&) {
    c->err = "zdwb_find_strings: out of host memory";
    return ZDWB_ERR_OOM;
  } catch (...) {
    c->err = "zdwb_find_strings: unexpected C++ exception";
    return ZDWB_ERR_CUDA;
  }
}

int zdwb_parse_numbers(zdwb_ctx* c, const zdwb_code_part* dict, const zdwb_number_opts* opts, zdwb_parse_out* out) {
  if (!c) return ZDWB_ERR_BAD_ARG;
  c->err.clear();
  if (!opts || !out) {
    c->err = "zdwb_parse_numbers: null argument";
    return ZDWB_ERR_BAD_ARG;
  }
  if (cudaSetDevice(c->device) != cudaSuccess) {
    c->err = "cudaSetDevice failed";
    return ZDWB_ERR_NO_DEVICE;
  }
  try {
    return zdwb::parse_numbers_impl(c, dict, opts, out);
  } catch (const std::bad_alloc&) {
    c->err = "zdwb_parse_numbers: out of host memory";
    return ZDWB_ERR_OOM;
  } catch (...) {
    c->err = "zdwb_parse_numbers: unexpected C++ exception";
    return ZDWB_ERR_CUDA;
  }
}

int zdwb_format_numbers(zdwb_ctx* c, const int64_t* values, uint64_t n, const zdwb_number_opts* opts, zdwb_merge_out* out) {
  if (!c) return ZDWB_ERR_BAD_ARG;
  c->err.clear();
  if (!opts || !out) {
    c->err = "zdwb_format_numbers: null argument";
    return ZDWB_ERR_BAD_ARG;
  }
  if (cudaSetDevice(c->device) != cudaSuccess) {
    c->err = "cudaSetDevice failed";
    return ZDWB_ERR_NO_DEVICE;
  }
  try {
    return zdwb::format_numbers_impl(c, values, n, opts, out);
  } catch (const std::bad_alloc&) {
    c->err = "zdwb_format_numbers: out of host memory";
    return ZDWB_ERR_OOM;
  } catch (...) {
    c->err = "zdwb_format_numbers: unexpected C++ exception";
    return ZDWB_ERR_CUDA;
  }
}

void* zdwb_host_alloc(size_t bytes) {
  void* p = nullptr;
  if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) {
    (void)cudaGetLastError();
    return nullptr;
  }
  return p;
}

void zdwb_host_free(void* p) {
  if (p) cudaFreeHost(p);
}

}  // extern "C"
