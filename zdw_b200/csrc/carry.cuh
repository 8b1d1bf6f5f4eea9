// carry.cuh -- "last explicit value per column" carried across strips of rows (used by the decoder for the
// reference's columnVal[] state, UnconvertFromZDW.cpp:985-986,1349-1453).
//
// Input: for every strip s and used column u, shas[s*U+u] = the strip holds an explicit value for the column and
// sval[s*U+u] = the last one.  Output: cin[s*U+u] = the value the column has where strip s begins (0 at block start).
// "Select the last explicit value" is associative: strips are grouped into segments of S, reduced, scanned, applied.
#pragma once
#include <stdint.h>

#include "common.cuh"

namespace zdwb {
namespace {

// carry propagation over strips, per used column: "select the last explicit value" is associative
__global__ void k_carry_reduce(const unsigned long long* __restrict__ sval, const uint8_t* __restrict__ shas,
                               uint32_t nstrips, uint32_t U, uint32_t S, unsigned long long* __restrict__ seg_val,
                               uint8_t* __restrict__ seg_has) {
  const uint32_t u = blockIdx.x * blockDim.x + threadIdx.x, seg = blockIdx.y;
  if (u >= U) return;
  const uint32_t sb = seg * S, se = min(nstrips, sb + S);
  unsigned long long v = 0;
  uint8_t h = 0;
  for (uint32_t s = sb; s < se; ++s) {
    if (shas[(size_t)s * U + u]) {
      v = sval[(size_t)s * U + u];
      h = 1;
    }
  }
  seg_val[(size_t)seg * U + u] = v;
  seg_has[(size_t)seg * U + u] = h;
}

__global__ void k_carry_scan(unsigned long long* __restrict__ seg_val, const uint8_t* __restrict__ seg_has, uint32_t nseg,
                             uint32_t U) {
  const uint32_t u = blockIdx.x * blockDim.x + threadIdx.x;
  if (u >= U) return;
  unsigned long long v = 0;  // columnVal starts at 0 in every block: UnconvertFromZDW.cpp:985-986
  for (uint32_t s = 0; s < nseg; ++s) {
    const unsigned long long mine = seg_val[(size_t)s * U + u];
    const uint8_t h = seg_has[(size_t)s * U + u];
    seg_val[(size_t)s * U + u] = v;  // becomes the carry-in of the segment
    if (h) v = mine;
  }
}

__global__ void k_carry_apply(const unsigned long long* __restrict__ sval, const uint8_t* __restrict__ shas,
                              const unsigned long long* __restrict__ seg_cin, uint32_t nstrips, uint32_t U, uint32_t S,
                              unsigned long long* __restrict__ cin) {
  const uint32_t u = blockIdx.x * blockDim.x + threadIdx.x, seg = blockIdx.y;
  if (u >= U) return;
  const uint32_t sb = seg * S, se = min(nstrips, sb + S);
  unsigned long long v = seg_cin[(size_t)seg * U + u];
  for (uint32_t s = sb; s < se; ++s) {
    cin[(size_t)s * U + u] = v;
    if (shas[(size_t)s * U + u]) v = sval[(size_t)s * U + u];
  }
}

// cin of nstrips strips of U used columns from their sval / shas: reduce, scan and apply over segments of S strips
int carry_prefix(Ctx* ctx, const unsigned long long* sval, const uint8_t* shas, uint32_t nstrips, uint32_t U,
                 unsigned long long* cin) {
  const uint32_t S = std::max<uint32_t>((nstrips + 255) / 256, 4);  // (the scan over segments is a serial loop: at least 4 per segment)
  const uint32_t nseg = (nstrips + S - 1) / S;
  DevBuf seg_val, seg_has;
  ZDWB_TRY(seg_val.alloc(ctx, (size_t)nseg * U * 8));
  ZDWB_TRY(seg_has.alloc(ctx, (size_t)nseg * U));
  const dim3 g2((U + 127) / 128, nseg);
  ZDWB_TRY(launch(ctx, "k_carry_reduce", k_carry_reduce, g2, 128, 0, sval, shas, nstrips, U, S, seg_val.as<unsigned long long>(),
                  seg_has.as<uint8_t>()));
  ZDWB_TRY(launch(ctx, "k_carry_scan", k_carry_scan, (U + 127) / 128, 128, 0, seg_val.as<unsigned long long>(),
                  seg_has.as<uint8_t>(), nseg, U));
  return launch(ctx, "k_carry_apply", k_carry_apply, g2, 128, 0, sval, shas, seg_val.as<unsigned long long>(), nstrips, U, S, cin);
}

}  // namespace
}  // namespace zdwb
