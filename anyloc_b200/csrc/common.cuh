// Shared helpers for libanyloc_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>
#include <math.h>
#include "../../include/anyloc_b200.h"

namespace anyloc {

void set_error(const char* fmt, ...);

#define ANYLOC_CHECK_CUDA(expr)                                                        \
  do {                                                                                 \
    cudaError_t _e = (expr);                                                           \
    if (_e != cudaSuccess) {                                                           \
      anyloc::set_error("%s:%d CUDA error %s: %s", __FILE__, __LINE__,                 \
                        cudaGetErrorName(_e), cudaGetErrorString(_e));                 \
      return ANYLOC_ERR_CUDA;                                                          \
    }                                                                                  \
  } while (0)

#define ANYLOC_CHECK_LAUNCH()                                                          \
  do {                                                                                 \
    anyloc::count_launch();                                                            \
    ANYLOC_CHECK_CUDA(cudaGetLastError());                                             \
  } while (0)

#define ANYLOC_REQUIRE(cond, ...)                                                      \
  do {                                                                                 \
    if (!(cond)) {                                                                     \
      anyloc::set_error(__VA_ARGS__);                                                  \
      return ANYLOC_ERR_ARG;                                                           \
    }                                                                                  \
  } while (0)

static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }
static inline int cdiv(int a, int b) { return (a + b - 1) / b; }

// bump allocator over a caller-owned workspace
struct Workspace {
  char* base; size_t size; size_t off;
  Workspace(void* p, size_t n) : base((char*)p), size(n), off(0) {}
  template <typename T> T* take(size_t count) {
    size_t bytes = align_up(count * sizeof(T), 256);
    if (off + bytes > size) return nullptr;
    T* r = (T*)(base + off); off += bytes; return r;
  }
};

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// fp32 -> (hi, lo): hi = round-to-nearest tf32 (10 explicit mantissa bits, low 13 bits zero),
// lo = x - hi (exact in fp32).  hi + lo == x exactly.
__device__ __forceinline__ void split_tf32(float x, float& hi, float& lo) {
  uint32_t u;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(x));
  hi = __uint_as_float(u & 0xffffe000u);
  lo = x - hi;
}

// fp16 pair format (engine TC3H): a GEMM input x is stored as (hi, lo) = (fp16(s*x), fp16(s*x - hi)), s a power
// of two; hi+lo carries ~22 significant bits of s*x like the tf32 pair, at half the bytes and on the 2x faster
// kind::f16 tensor path.  Activations use the fixed scale kActScale, weights a per-tensor scale (see vit.py);
// the GEMM epilogue multiplies the accumulator by alpha = 1/(s_A*s_B) (exact).
constexpr float kActScale = 8.0f;
// f32 <-> f16 conversions run on the 16-lane/clk conversion path (measured: they, not the FMAs, bounded the softmax
// warps of the attention kernel), so the hi part is rounded to 11 significant bits with Veltkamp's splitting on the
// FMA pipe (t = x*(2^13+1); hi = t - (t - x), round-to-nearest) and only the final packs use cvt -- one
// cvt.rn.f16x2.f32 per TWO elements in the packed variant.
__device__ __forceinline__ float veltkamp_hi11(float x) {
  const float t = __fmul_rn(x, 8193.0f);
  return __fsub_rn(t, __fsub_rn(t, x));
}
__device__ __forceinline__ void split_f16(float xs, __half& hi, __half& lo) {
  const float h = veltkamp_hi11(xs);
  hi = __float2half_rn(h);                       // exact (11 significant bits) inside the fp16 normal range
  lo = __float2half_rn(__fsub_rn(xs, h));
}
// two values -> packed (hi, lo) words; `a` lands in the low 16 bits (element k), `b` in the high 16 bits (k+1)
__device__ __forceinline__ void split_f16x2(float a, float b, uint32_t& hi2, uint32_t& lo2) {
  const float ha = veltkamp_hi11(a), hb = veltkamp_hi11(b);
  const float la = __fsub_rn(a, ha), lb = __fsub_rn(b, hb);
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(hi2) : "f"(hb), "f"(ha));
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(lo2) : "f"(lb), "f"(la));
}

int device_sm_count();
// true the first time it is called on the CURRENT device for this flag word: cudaFuncSetAttribute is per device, so a
// process that drives several GPUs must repeat it on each of them (one bit per device ordinal; atomic because two host
// threads may race on the word).  A failing cudaFuncSetAttribute is reported to the caller by ANYLOC_CHECK_CUDA; the
// launch that follows a failed attribute set fails loudly as well (dynamic shared memory over the default limit).
static inline bool first_use_on_this_device(unsigned long long* seen) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return true;
  const unsigned long long bit = 1ull << dev;
  const unsigned long long old = __atomic_fetch_or(seen, bit, __ATOMIC_RELAXED);
  return (old & bit) == 0;
}
void count_launch();

// Optional per-category device timing (cudaEvents on the launching stream), see anyloc_profile_*.
enum ProfCat { PC_GEMM_TC = 0, PC_GEMM_SIMT, PC_ATTENTION, PC_LAYERNORM, PC_VIT_MISC, PC_VLAD, PC_TOPK, PC_LOG_BIN,
               PC_COUNT };
struct ProfScope {
  int slot; cudaStream_t st;
  ProfScope(int cat, cudaStream_t stream, double work);
  ~ProfScope();
};

}  // namespace anyloc
