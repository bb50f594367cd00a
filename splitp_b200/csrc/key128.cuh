// 128-bit pattern keys {lo, hi} (up to 64 taxa) and their hash-table primitives, shared by wide.cu and mi_batch.cu.
// The all-ones key is the EMPTY marker of every table built from these.
#pragma once
#include "common.cuh"

namespace spb {

constexpr unsigned long long kAll = 0xFFFFFFFFFFFFFFFFull;

struct Key128 {
  unsigned long long lo, hi;
};

__device__ __forceinline__ bool is_empty(Key128 k) { return k.lo == kAll && k.hi == kAll; }
__device__ __forceinline__ bool same(Key128 a, Key128 b) { return a.lo == b.lo && a.hi == b.hi; }

// plain 16-byte read: only used by kernels that run after all insertions have completed
__device__ __forceinline__ Key128 load_key(const unsigned long long* keys, uint64_t slot) {
  const ulonglong2 v = *reinterpret_cast<const ulonglong2*>(keys + 2 * slot);
  return Key128{v.x, v.y};
}

__device__ __forceinline__ Key128 cas128(unsigned long long* ptr, Key128 cmp, Key128 val) {
  Key128 old;
  asm volatile(
      "{\n\t.reg .b128 c, v, o;\n\t"
      "mov.b128 c, {%2, %3};\n\t"
      "mov.b128 v, {%4, %5};\n\t"
      "atom.global.cas.b128 o, [%6], c, v;\n\t"
      "mov.b128 {%0, %1}, o;\n\t}"
      : "=l"(old.lo), "=l"(old.hi)
      : "l"(cmp.lo), "l"(cmp.hi), "l"(val.lo), "l"(val.hi), "l"(ptr)
      : "memory");
  return old;
}

__device__ __forceinline__ uint64_t hash128(Key128 k) { return mix64(k.lo ^ mix64(k.hi + 0x9E3779B97F4A7C15ull)); }

}  // namespace spb
