// Shared device/host helpers for the coda_b200 kernels (sm_100a only).
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <math.h>

#include "../../include/coda_b200.h"

#define CODA_WARP 32
#define CODA_FULL 0xffffffffu

// ---- error plumbing (thread-local message, C-ABI returns an int code) -----------------
void coda_set_error(const char* fmt, ...);

#define CODA_CHECK_ARG(cond, ...)                                   \
  do {                                                              \
    if (!(cond)) {                                                  \
      coda_set_error(__VA_ARGS__);                                  \
      return CODA_B200_EINVAL;                                      \
    }                                                               \
  } while (0)

#define CODA_CUDA_OK(expr)                                                        \
  do {                                                                            \
    cudaError_t _e = (expr);                                                      \
    if (_e != cudaSuccess) {                                                      \
      coda_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),      \
                     __FILE__, __LINE__);                                         \
      return CODA_B200_ECUDA;                                                     \
    }                                                                             \
  } while (0)

#define CODA_LAUNCH_OK(name)                                                      \
  do {                                                                            \
    cudaError_t _e = cudaGetLastError();                                          \
    if (_e != cudaSuccess) {                                                      \
      coda_set_error("launch of %s failed: %s", name, cudaGetErrorString(_e));    \
      return CODA_B200_ECUDA;                                                     \
    }                                                                             \
  } while (0)

static inline cudaStream_t as_stream(coda_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }

int coda_sm_count();   // cached multiprocessor count of the current device

// ---- warp primitives -----------------------------------------------------------------
template <typename T>
__device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(CODA_FULL, v, o);
  return v;
}

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(CODA_FULL, v, o));
  return v;
}

// (value, index) arg-max with "first index wins" on equal values (torch.argmax on CPU).
__device__ __forceinline__ void warp_argmax(float& v, int& i) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    float ov = __shfl_xor_sync(CODA_FULL, v, o);
    int oi = __shfl_xor_sync(CODA_FULL, i, o);
    if (ov > v || (ov == v && oi < i)) { v = ov; i = oi; }
  }
}

// ---- entropy term, coda.py:254/276: f(m) = -max(m,1e-12) * log2(max(m,1e-12)) ----------
// MUFU.LG2 (abs error <= 2^-22 on [0.5, 2], 2 ulp elsewhere; q is never denormal): the gain sums
// differences of these terms and stays ~1e-8 accurate, far inside the 5e-6 EIG parity budget.
__device__ __forceinline__ float ent_term(float m) {
  float q = fmaxf(m, 1e-12f);
  return -q * __log2f(q);
}

// ---- row normalisation, coda.py:230-231: xi = u / den for every entry of a row ----------------------------
// One IEEE division per row (rden = 1 / den), then per entry the Markstein correction  q = u rden,  q += (u - den q) rden,
// which returns the correctly rounded quotient (the same bits as u / den, except for the measure-zero case of a den
// whose significand is all ones) in 3 instructions instead of the ~20 of the division subroutine: at C = 1000 the
// row pass was instruction-bound on it.  EVERY kernel that normalises rows of U goes through this function, so the
// column sums of the full pass, of every rank-1 variant and of a resumed run stay bit-identical to each other.
__device__ __forceinline__ float row_quot(float u, float den, float rden) {
  const float q = u * rden;
  return fmaf(fmaf(-den, q, u), rden, q);
}

// ---- fixed-point accumulation (order- and shard-count-independent sums) ---------------
// Values in [0, 1] are scaled by 2^shift and summed as int64; the host picks shift so that
// N_global * 2^shift < 2^62.
// `scale` = 2^shift as a float: v * scale is exact in fp32 (power-of-two scaling), so one F2I suffices.
__device__ __forceinline__ long long to_fx(float v, float scale) {
  return __float2ll_rn(v * scale);
}
__host__ __device__ __forceinline__ double from_fx(long long v, int shift) {
  return ldexp((double)v, -shift);
}

// ---- 1-D bulk TMA (cp.async.bulk, SASS UBLKCP) + mbarrier -------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"   // suspend-time hint: the hardware parks the warp
      "@p bra DONE;\n\t"                                                   // instead of spinning on the issue slots
      "bra WAIT_LOOP;\n\t"
      "DONE:\n\t"
      "}" ::"r"(smem_u32(bar)),
      "r"(parity), "r"(20000u)
      : "memory");
}
// global -> shared bulk copy; bytes % 16 == 0, both addresses 16-byte aligned.
__device__ __forceinline__ void tma_load_1d(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(smem_dst)),
      "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

// ---- slab element type: fp32, or IEEE binary16 (`__half`) converted on load -------------------------------------
// Every kernel that reads the prediction slab computes in fp32.  The fp16 -> fp32 conversion is exact, so a kernel
// instantiated for a 16-bit slab does the same arithmetic, with the same bits, as its fp32 twin on the upcast slab.
__device__ __forceinline__ float slab_ld(const float* p) { return __ldg(p); }
__device__ __forceinline__ float slab_ld(const __half* p) { return __half2float(__ldg(p)); }
__device__ __forceinline__ float slab_f(float v) { return v; }
__device__ __forceinline__ float slab_f(__half v) { return __half2float(v); }

// Bulk copies of 16-bit slab ranges: the range's start and length need not be 16-byte aligned, so the 16-byte aligned
// window around it is copied and the range starts `slab_head` bytes into the window.  The window stays inside the
// 16-byte granules of the allocation (device allocations are at least 256-byte aligned and sized).  Shared-memory
// buffers that receive such a window carry SLAB_PAD bytes of slack.  An fp32 range is copied as is (callers guarantee
// its alignment), so the fp32 instantiations issue exactly the copies they always did.
template <typename T>
__host__ __device__ constexpr uint32_t slab_pad() { return sizeof(T) == 4 ? 0u : 16u; }
template <typename T>
__device__ __forceinline__ uint32_t slab_head(const T* p) {
  return sizeof(T) == 4 ? 0u : (uint32_t)(reinterpret_cast<uintptr_t>(p) & 15);
}
template <typename T>
__device__ __forceinline__ uint32_t tma_load_slab(void* smem_dst, const T* src, uint32_t bytes, uint64_t* bar) {
  const uint32_t head = slab_head(src);
  const uint32_t win = sizeof(T) == 4 ? bytes : ((head + bytes + 15u) & ~15u);
  mbar_expect_tx(bar, win);
  tma_load_1d(smem_dst, reinterpret_cast<const unsigned char*>(src) - head, win, bar);
  return head;
}

// ---- arg-max records ---------------------------------------------------------------------------
// One record = CODA_B200_REC_WORDS int64: {bits(vA), iA, cntA, bits(vB), iB, bits(v2A), bits(v2B), 0}.
//   set A = unlabeled & non-unanimous items (coda.py:215-219), set B = all unlabeled items (coda.py:239 fallback);
//   v / i = best value and its lowest global index (torch.argmax: first maximum, coda.py:309), cnt = |A|,
//   v2 = best value among the OTHER items of the set (for the isclose tie test of coda.py:307).
#define IDX_NONE 0x7fffffffffffffffLL
#define REC_W CODA_B200_REC_WORDS

struct Best2 {
  float v;
  long long i;
  float v2;
};
__device__ __forceinline__ Best2 best2_empty() { return Best2{-INFINITY, IDX_NONE, -INFINITY}; }
__device__ __forceinline__ void best2_add(Best2& b, float v, long long i) {
  if (v > b.v || (v == b.v && i < b.i)) {
    b.v2 = fmaxf(b.v2, b.v);
    b.v = v;
    b.i = i;
  } else {
    b.v2 = fmaxf(b.v2, v);
  }
}
__device__ __forceinline__ void best2_merge(Best2& b, const Best2& o) {
  if (o.i == IDX_NONE) return;
  if (b.i == IDX_NONE) { b = o; return; }
  if (o.v > b.v || (o.v == b.v && o.i < b.i)) {
    const float lose = b.v;
    b.v2 = fmaxf(fmaxf(b.v2, o.v2), lose);
    b.v = o.v;
    b.i = o.i;
  } else {
    b.v2 = fmaxf(fmaxf(b.v2, o.v2), o.v);
  }
}
__device__ __forceinline__ void best2_warp(Best2& b) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    Best2 t;
    t.v = __shfl_xor_sync(CODA_FULL, b.v, o);
    t.i = __shfl_xor_sync(CODA_FULL, b.i, o);
    t.v2 = __shfl_xor_sync(CODA_FULL, b.v2, o);
    best2_merge(b, t);
  }
}
__device__ __forceinline__ void rec_store(long long* out, const Best2& a, long long cntA, const Best2& b) {
  out[0] = (long long)__float_as_int(a.v); out[1] = a.i; out[2] = cntA;
  out[3] = (long long)__float_as_int(b.v); out[4] = b.i;
  out[5] = (long long)__float_as_int(a.v2); out[6] = (long long)__float_as_int(b.v2); out[7] = 0;
}
__device__ __forceinline__ void rec_load(const long long* r, Best2& a, long long& cntA, Best2& b) {
  a.v = __int_as_float((int)r[0]); a.i = r[1]; cntA = r[2];
  b.v = __int_as_float((int)r[3]); b.i = r[4];
  a.v2 = __int_as_float((int)r[5]); b.v2 = __int_as_float((int)r[6]);
}
// torch.isclose(q, best, rtol=1e-8) with the default atol=1e-8, evaluated in fp32 (coda.py:307)
__device__ __forceinline__ bool isclose_best(float q, float best) {
  return q == best || fabsf(q - best) <= 1e-8f + fabsf(1e-8f * best);
}
