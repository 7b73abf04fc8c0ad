// pi_full on the 5th-generation tensor cores:  U[n][c] = sum_h sum_s preds[h][n][s] * D[h][c][s]   (coda.py:227-229)
//
// A skinny GEMM: M = N items, N = C classes, K = H*C.  One CTA owns a tile of 128 items and walks the H models; per model
// the 128 x C block of the slab is ONE contiguous blob (51 KB at C = 100), fetched by four 1-D bulk TMA copies.  fp32 does
// not go through tcgen05, so both operands are cut into two fp16 limbs, x = hi + 2^-12 lo  (11 + 11 significant bits: 2^-22
// relative at worst, a quarter of an fp32 ulp on average; lo is stored scaled so that it stays a normal fp16 number),
// and three products are formed per K = 16 chunk:
//
//     main  += A_hi . B_hi                    (22-bit products: exact in the fp32 accumulator)
//     corr  += A_hi . B_lo + A_lo . B_hi      (carries the 2^12 scale; A_lo . B_lo ~ 2^-22 is dropped)
//
// preds lie in [0, 1]; D (Dirichlet parameters) is multiplied by a power of two chosen from max |D| so that it stays
// inside the fp16 range, and U is scaled back at the end (exact).  The tensor core accumulates in fp32 with truncation,
// which biases a long chain of positive terms; so the two TMEM accumulators are drained every G (= 4) models into fp32
// registers (round-to-nearest adds) by dedicated warps, double-buffered so the drain of one group overlaps the MMAs of
// the next.  Against an fp64 contraction the result is closer than the 25 600-term fp32 FMA chain of the SIMT kernel
// (slab.cu: k_pi_full), see tests/test_gpu_parity.py::test_tensor_core_marginals_match_fp64.
//
// Roles (1024 threads x 64 registers, one CTA per SM):
//   warp 0 lane 0     slab producer     bulk TMA of (model, 32-item quarter) fp32 blocks into a staging ring
//   warp 1 lane 0     D producer        bulk TMA of the D limbs (pre-packed by k_pi_w_limbs), one K chunk per ring slot
//   warp 2            MMA issuer        per chunk A_hi . [D_hi | D_lo] (N = 2 Np: main | corr) and A_lo . D_hi (N = Np, into corr),
//                                       one tcgen05.commit per chunk frees its A and D slots
//   warps 4..19       drain             tcgen05.ld of both accumulators every G models, final store of U
//   warps 20..31      converters        fp32 staging -> fp16 hi / lo limbs in the UMMA K-major core-matrix order
//
// An fp16 slab (k_pi_full_tc<__half>) is staged as fp16, half the bytes per unit.  Its values ARE their own hi limb and
// their lo limb is exactly 0 (the split of the fp32 upcast gives the same two limbs), so the converters only repack the
// fp16 items into the core-matrix order; the lo limbs of the A ring are zeroed once and every MMA is issued as for fp32:
// the result has the bits of the fp32 pass on the upcast slab.  Its units are copied as 16-byte aligned windows
// (common.cuh: tma_load_slab), so an item-range view or an odd N needs no alignment beyond 8 bytes.
// The kernel lives on bytes in flight: every (tile, model) pulls 51 KB of slab from HBM and 50 KB of D limbs from L2, so
// shared memory is split between the fp32 staging ring and a deep D ring; the converted A chunks only need a short ring.
// Every wait is bounded: a pipeline that stops sets CODA_B200_FLAG_PIPELINE_TIMEOUT and the kernel drains out.
#include "common.cuh"

#include <cuda_fp16.h>
#include <stdlib.h>

namespace {

constexpr int PT_M = 128;                 // items per tile
constexpr int PT_THREADS = 1024;          // 32 warps x 64 registers: the whole register file
constexpr int PT_DRAIN_WARP0 = 4, PT_DRAIN_WARPS = 16;   // 4 lane quadrants x 4 column parts (<= 32 accumulator registers each)
constexpr int PT_DRAIN_PARTS = PT_DRAIN_WARPS / 4;
constexpr int PT_CONV_WARP0 = 20, PT_CONV_WARPS = 12;
constexpr int PT_WARPS_PER_CHUNK = 4;     // converter warps that share one K chunk (32 items each)
constexpr int PT_CONV_GROUPS = PT_CONV_WARPS / PT_WARPS_PER_CHUNK;
constexpr int PT_HALF = PT_M / PT_WARPS_PER_CHUNK;   // items per staging unit: one converter warp's share of a chunk
constexpr int PT_MAX_STAGES = 12;         // staging units
constexpr int PT_MAX_DSLOTS = 16;         // D chunks in flight (<= PT_CHUNK_BARS)
constexpr int PT_CHUNK_BARS = 16;         // per-chunk barriers, indexed by chunk number & 15 (power of two)
constexpr int PT_NBAR = 2 * PT_MAX_STAGES + 2 * PT_CHUNK_BARS + 4;
constexpr float PT_LO_SCALE = 4096.f;     // lo limbs are stored times 2^12
constexpr long long PT_TIMEOUT_CYCLES = 4000000000LL;   // ~2 s

struct PiTcArgs {
  const void* preds;          // float or __half [H][N][C]
  long long ldh;              // elements between models
  const unsigned char* wb;    // [H][KC][2 k_cores][2 Np/8 (hi | lo)][8][8] fp16, then the 16-byte header (max |D| bits)
  const uint32_t* dmax;       // header: bits of max |D|
  float* U;
  uint32_t* flags;
  long long N;
  int H, C, Np, KC;
  int NST, SA, SD;            // ring depths: staging units, converted A chunks, D chunks
  int G;                      // models per accumulator drain
};

// power of two that brings max |D| below 2^15 (fp16 overflows at 65504); 0 when no scaling is needed
__device__ __forceinline__ int pt_down_shift(uint32_t maxbits) {
  const int e = (int)((maxbits >> 23) & 0xffu) - 127;
  return max(0, e - 14);
}

__device__ __forceinline__ void pt_fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void pt_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void pt_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void pt_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// one lane of a converged warp
__device__ __forceinline__ bool pt_elect() {
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "elect.sync _|P, 0xFFFFFFFF;\n\t"
      "selp.b32 %0, 1, 0, P;\n\t"
      "}"
      : "=r"(pred));
  return pred != 0;
}

// try_wait with a suspend-time hint: the warp is parked by the hardware until the phase completes (or ~the hint elapses)
// instead of burning the issue slots the converter warps need
__device__ __forceinline__ bool pt_try(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity), "r"(20000u)
      : "memory");
  return ok != 0;
}

// false = the pipeline was aborted (here or by another role)
__device__ __forceinline__ bool pt_wait(uint64_t* bar, uint32_t parity, volatile int* abort_s) {
  if (pt_try(bar, parity)) return true;
  const long long t0 = clock64();
  for (;;) {
    if (pt_try(bar, parity)) return true;
    if (*abort_s) return false;
    if (clock64() - t0 > PT_TIMEOUT_CYCLES) {
      *abort_s = 1;
      return false;
    }
  }
}

// a position in a ring of `n` slots walked one or several steps at a time; `ph` = parity of the number of wraps
struct Ring {
  int slot, ph, wrapped;
  __device__ __forceinline__ void step(int by, int n) {
    slot += by;
    while (slot >= n) { slot -= n; ph ^= 1; wrapped = 1; }
  }
};

// cute::UMMA::SmemDescriptor words (SWIZZLE_NONE, K-major, see pairs_tc.cu) are assembled in the MMA warp
__device__ __forceinline__ uint64_t pt_pack(uint32_t lo, uint32_t hi) {
  uint64_t d;
  asm("mov.b64 %0, {%1, %2};" : "=l"(d) : "r"(lo), "r"(hi));
  return d;
}
// cute::UMMA::InstrDescriptor: c = F32 (1) [4,6), a = b = F16 (0) [7,10) [10,13), K-major both, N >> 3 [17,23), M >> 4 [24,29)
__device__ __forceinline__ uint32_t pt_idesc(int n) {
  return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(PT_M >> 4) << 24);
}
__device__ __forceinline__ void pt_mma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum)
      : "memory");
}
__device__ __forceinline__ void pt_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void pt_tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// two floats -> packed fp16 hi limbs and packed fp16 lo limbs:  x = hi + lo / 4096 (+ 2^-22 x at worst)
__device__ __forceinline__ void pt_split2(float a, float b, uint32_t& hi, uint32_t& lo) {
  const __half2 h = __floats2half2_rn(a, b);
  const float2 hf = __half22float2(h);
  const __half2 l = __floats2half2_rn((a - hf.x) * PT_LO_SCALE, (b - hf.y) * PT_LO_SCALE);   // a - hi is exact
  hi = *reinterpret_cast<const uint32_t*>(&h);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}

// ---- max |D| (bit pattern; D is finite and positive in every valid run, NaN / Inf end up as NaN in U) ---------------
__global__ void __launch_bounds__(256) k_pi_w_max(const float* __restrict__ D, long long n, uint32_t* __restrict__ out) {
  uint32_t m = 0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    m = max(m, __float_as_uint(fabsf(D[i])));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(CODA_FULL, m, o));
  if ((threadIdx.x & 31) == 0 && m) atomicMax(out, m);
}

// ---- D -> fp16 limbs in the B-operand order: one blob per (model, K chunk) -----------------------------------------
// blob = [k_core 2][n_core 2 Np/8: hi limbs, then lo limbs][8 classes][8 s] fp16;  class = n_core*8 + r,  s = chunk*16 + k_core*8 + e
// (hi and lo side by side along N, so that A_hi . [D_hi | D_lo] is ONE tcgen05.mma of N = 2 Np)
__global__ void __launch_bounds__(256) k_pi_w_limbs(const float* __restrict__ D, int H, int C, int Np, int KC,
                                                    const uint32_t* __restrict__ dmax, __half* __restrict__ wb) {
  const long long per_limb = (long long)2 * Np * 8;           // elements of one limb of one chunk (= Np x 16)
  const long long total = (long long)H * KC * per_limb;
  const float down = __uint_as_float((uint32_t)(127 - pt_down_shift(*dmax)) << 23);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int e = (int)(i & 7), r = (int)((i >> 3) & 7);
    long long q = i >> 6;
    const int ncore = (int)(q % (Np / 8));
    q /= (Np / 8);
    const int kcore = (int)(q & 1);
    q >>= 1;
    const int kc = (int)(q % KC);
    const int h = (int)(q / KC);
    const int c = ncore * 8 + r, s = kc * 16 + kcore * 8 + e;
    const float v = (c < C && s < C) ? D[((size_t)h * C + c) * C + s] * down : 0.f;
    const __half hi = __float2half_rn(v);
    const __half lo = __float2half_rn((v - __half2float(hi)) * PT_LO_SCALE);
    const long long blob = ((long long)h * KC + kc) * 2 * per_limb;
    const long long within = ((long long)kcore * (2 * Np / 8) + ncore) * 64 + r * 8 + e;
    wb[blob + within] = hi;
    wb[blob + (long long)(Np / 8) * 64 + within] = lo;
  }
}

template <typename T>
__global__ void __launch_bounds__(PT_THREADS, 1) k_pi_full_tc(PiTcArgs a) {
  extern __shared__ __align__(1024) unsigned char smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int H = a.H, C = a.C, Np = a.Np, KC = a.KC, NST = a.NST, SA = a.SA, SD = a.SD, G = a.G;
  const long long n0 = (long long)blockIdx.x * PT_M;
  const int cnt = (int)min((long long)PT_M, a.N - n0);

  // ---- shared memory carve-up ----------------------------------------------------------------------
  const T* preds = reinterpret_cast<const T*>(a.preds);
  const uint32_t stage_bytes = (uint32_t)PT_HALF * C * sizeof(T) + slab_pad<T>();   // block of one (model, 32-item quarter)
  const uint32_t stage_stride = (stage_bytes + 127u) & ~127u;
  const uint32_t a_limb = (uint32_t)PT_M * 16u * 2u;                          // 4 KB: one limb of one A chunk
  const uint32_t b_limb = (uint32_t)Np * 16u * 2u;                            // one limb of one D chunk
  unsigned char* stage0 = smem;
  unsigned char* aslots = smem + (uint32_t)NST * stage_stride;                // [SA][2 limbs]
  unsigned char* dslots = aslots + (uint32_t)SA * 2u * a_limb;                // [SD][2 limbs]
  unsigned char* tail = dslots + (uint32_t)SD * 2u * b_limb;
  uint64_t* fullS = reinterpret_cast<uint64_t*>(tail);        // staging unit filled (TMA)
  uint64_t* emptyS = fullS + PT_MAX_STAGES;                   // staging unit consumed (its converter warps)
  uint64_t* fullK = emptyS + PT_MAX_STAGES;                   // chunk q ready (index q & 15): 2 converter warps + the D TMA
  uint64_t* doneK = fullK + PT_CHUNK_BARS;                    // chunk q consumed (index q & 15): tcgen05.commit
  uint64_t* accFull = doneK + PT_CHUNK_BARS;                  // [2] accumulator group complete (tcgen05.commit)
  uint64_t* accEmpty = accFull + 2;                           // [2] accumulator drained (drain warps)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(accEmpty + 2);
  volatile int* abort_s = reinterpret_cast<volatile int*>(tmem_slot + 1);

  if (tid == 0) {
    for (int i = 0; i < PT_MAX_STAGES; ++i) {
      mbar_init(&fullS[i], 1);
      mbar_init(&emptyS[i], PT_CONV_GROUPS);
    }
    for (int i = 0; i < PT_CHUNK_BARS; ++i) {
      mbar_init(&fullK[i], PT_WARPS_PER_CHUNK + 1);
      mbar_init(&doneK[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&accFull[i], 1);
      mbar_init(&accEmpty[i], PT_DRAIN_WARPS);
    }
    *abort_s = (*a.flags & CODA_B200_FLAG_PIPELINE_TIMEOUT) ? 1 : 0;          // an earlier CTA already gave up
    mbar_fence_init();
  }
  if constexpr (sizeof(T) == 2) {                                              // fp16 slab: the lo limbs of A are 0
    for (uint32_t i = tid; i < (uint32_t)SA * (a_limb / 16u); i += PT_THREADS) {
      const uint32_t s = i / (a_limb / 16u), e = i % (a_limb / 16u);
      *reinterpret_cast<uint4*>(aslots + (size_t)s * 2u * a_limb + a_limb + e * 16u) = make_uint4(0u, 0u, 0u, 0u);
    }
    pt_fence_proxy_async();                                                    // visible to the tensor core
  }
  if (warp == 3) {
    __syncwarp();
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  pt_fence_before();
  __syncthreads();
  pt_fence_after();
  const uint32_t tmem = *tmem_slot;
  const int total_chunks = H * KC;
  const int ngroups = (H + G - 1) / G;

  if (warp == 0) {
    // ---- slab producer: unit j = (model j / 4, 32-item quarter j % 4) ----------------------------------------
    if (lane == 0) {
      Ring r{0, 0, 0};
      for (int j = 0; j < PT_WARPS_PER_CHUNK * H; ++j, r.step(1, NST)) {
        const int hf = j % PT_WARPS_PER_CHUNK;
        if (r.wrapped && !pt_wait(&emptyS[r.slot], r.ph ^ 1, abort_s)) break;
        const int items = min(PT_HALF, max(0, cnt - hf * PT_HALF));
        if (items == 0) {                                     // ragged last tile: nothing in this half
          pt_arrive(&fullS[r.slot]);
          continue;
        }
        const uint32_t bytes = (uint32_t)items * C * sizeof(T);
        tma_load_slab(stage0 + (size_t)r.slot * stage_stride,
                      preds + (size_t)(j / PT_WARPS_PER_CHUNK) * a.ldh + (size_t)(n0 + hf * PT_HALF) * C, bytes, &fullS[r.slot]);
      }
    }
  } else if (warp == 1) {
    // ---- D producer ---------------------------------------------------------------------------------
    if (lane == 0) {
      const uint32_t bytes = 2u * b_limb;
      Ring r{0, 0, 0};
      for (int q = 0; q < total_chunks; ++q, r.step(1, SD)) {
        const int w = q - SD;                                 // the chunk that held this slot
        if (w >= 0 && !pt_wait(&doneK[w & (PT_CHUNK_BARS - 1)], (w / PT_CHUNK_BARS) & 1, abort_s)) break;
        uint64_t* full = &fullK[q & (PT_CHUNK_BARS - 1)];
        mbar_expect_tx(full, bytes);
        tma_load_1d(dslots + (size_t)r.slot * bytes, a.wb + (size_t)q * bytes, bytes, full);
      }
    }
  } else if (warp == 2) {
    // ---- MMA issuer: the whole warp walks the loop (so everything stays in uniform registers), one elected lane issues.
    // The issue rate of this one warp bounds the tensor pipe (an MMA of N = 112 is 56 cycles), so ring positions and
    // descriptors are stepped incrementally: no division, no descriptor rebuild per chunk.
    {
      const uint32_t tmem_u = __shfl_sync(CODA_FULL, tmem, 0);
      const uint32_t idesc2 = pt_idesc(2 * Np), idesc1 = pt_idesc(Np);
      // descriptor words (SWIZZLE_NONE, K-major): lo = start >> 4 | LBO >> 4 << 16, hi = SBO >> 4 | version 1 << 14
      const uint32_t a_lo0 = ((smem_u32(aslots) & 0x3FFFFu) >> 4) | ((uint32_t)((PT_M / 8) * 128 >> 4) << 16);
      const uint32_t d_lo0 = ((smem_u32(dslots) & 0x3FFFFu) >> 4) | ((uint32_t)((2 * Np / 8) * 128 >> 4) << 16);
      const uint32_t desc_hi = (128u >> 4) | (1u << 14);
      const uint32_t a_step = (2u * a_limb) >> 4, a_limb16 = a_limb >> 4, d_step = (2u * b_limb) >> 4;
      uint32_t a_off = 0, d_off = 0, kph = 0;
      int a_slot = 0, d_slot = 0, bi = 0;
      bool ok = true;
      for (int g = 0; g < ngroups && ok; ++g) {
        const int buf = g & 1;
        if (g >= 2) {
          ok = pt_wait(&accEmpty[buf], ((g >> 1) - 1) & 1, abort_s);
          ok = __all_sync(CODA_FULL, ok);
          if (!ok) break;
          pt_fence_after();
        }
        const uint32_t t_main = tmem_u + (uint32_t)buf * 256u, t_corr = t_main + (uint32_t)Np;
        const int nchunks = (min(H, (g + 1) * G) - g * G) * KC;
        for (int k = 0; k < nchunks; ++k) {
          ok = pt_wait(&fullK[bi], kph, abort_s);
          ok = __all_sync(CODA_FULL, ok);
          if (!ok) break;
          pt_fence_after();
          if (pt_elect()) {
            const uint64_t d_all = pt_pack(d_lo0 + d_off, desc_hi);
            pt_mma(t_main, pt_pack(a_lo0 + a_off, desc_hi), d_all, idesc2, k ? 1u : 0u);     // [main | corr] (+)= A_hi . [D_hi | D_lo]
            pt_mma(t_corr, pt_pack(a_lo0 + a_off + a_limb16, desc_hi), d_all, idesc1, 1u);    // corr += A_lo . D_hi
            pt_commit(&doneK[bi]);
          }
          __syncwarp();
          a_off += a_step;
          if (++a_slot == SA) { a_slot = 0; a_off = 0; }
          d_off += d_step;
          if (++d_slot == SD) { d_slot = 0; d_off = 0; }
          if (++bi == PT_CHUNK_BARS) { bi = 0; kph ^= 1u; }
        }
        if (ok && pt_elect()) pt_commit(&accFull[buf]);
        __syncwarp();
      }
    }
  } else if (warp >= PT_DRAIN_WARP0 && warp < PT_DRAIN_WARP0 + PT_DRAIN_WARPS) {
    // ---- drain: (item, column part) per thread: lane quadrant = warp % 4 (hardware rule), 16-column units u_lo..u_hi -----
    const int quad = warp & 3, part = (warp - PT_DRAIN_WARP0) >> 2;
    const int row = quad * 32 + lane;
    const int nu = Np / 16;                                   // 16-column units (<= 8)
    const int per = (nu + PT_DRAIN_PARTS - 1) / PT_DRAIN_PARTS;               // <= 2 units per thread
    const int u_lo = min(nu, part * per), u_hi = min(nu, u_lo + per);
    float acc[2][16];
#pragma unroll
    for (int u = 0; u < 2; ++u)
#pragma unroll
      for (int i = 0; i < 16; ++i) acc[u][i] = 0.f;
    bool ok = true;
    for (int g = 0; g < ngroups; ++g) {
      const int buf = g & 1;
      ok = pt_wait(&accFull[buf], (g >> 1) & 1, abort_s);
      ok = __all_sync(CODA_FULL, ok);
      if (!ok) break;
      pt_fence_after();
      const uint32_t trow = tmem + ((uint32_t)(quad * 32) << 16) + (uint32_t)buf * 256u;
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        if (u_lo + u < u_hi) {                                // warp-uniform
          float m[16];
          pt_tmem_ld16(trow + (uint32_t)(u_lo + u) * 16u, m);
#pragma unroll
          for (int i = 0; i < 16; ++i) acc[u][i] += m[i];
          pt_tmem_ld16(trow + (uint32_t)Np + (uint32_t)(u_lo + u) * 16u, m);
#pragma unroll
          for (int i = 0; i < 16; ++i) acc[u][i] = fmaf(m[i], 1.0f / PT_LO_SCALE, acc[u][i]);
        }
      }
      pt_fence_before();
      __syncwarp();
      if (lane == 0) pt_arrive(&accEmpty[buf]);
    }
    if (ok && row < cnt) {
      const float up = __uint_as_float((uint32_t)(127 + pt_down_shift(*a.dmax)) << 23);      // undo the D range scaling
      float* urow = a.U + (size_t)(n0 + row) * C;
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        if (u_lo + u < u_hi) {
          const int c0 = (u_lo + u) * 16;
#pragma unroll
          for (int i = 0; i < 16; i += 4)
            if (c0 + i < C)                                   // C % 4 == 0: whole float4 in range
              *reinterpret_cast<float4*>(urow + c0 + i) =
                  make_float4(acc[u][i] * up, acc[u][i + 1] * up, acc[u][i + 2] * up, acc[u][i + 3] * up);
        }
      }
    }
  } else if (warp >= PT_CONV_WARP0) {
    // ---- converters: warp pair `grp` takes chunks q = grp, grp + PT_CONV_GROUPS, ...; `sub` picks the 32-item quarter ------
    const int cw = warp - PT_CONV_WARP0;
    const int grp = cw / PT_WARPS_PER_CHUNK, sub = cw % PT_WARPS_PER_CHUNK;
    bool ok = true;
    int q = grp;                                              // this warp's next chunk (global chunk index)
    Ring rs{0, 0, 0}, ra{0, 0, 0};
    rs.step(sub, NST);                                        // staging unit PT_WARPS_PER_CHUNK * h + sub
    ra.step(grp, SA);
    for (int h = 0; h < H && ok; ++h, rs.step(PT_WARPS_PER_CHUNK, NST)) {
      ok = pt_wait(&fullS[rs.slot], rs.ph, abort_s);
      ok = __all_sync(CODA_FULL, ok);
      if (!ok) break;
      const unsigned char* stage = stage0 + (size_t)rs.slot * stage_stride;
      const float* src = reinterpret_cast<const float*>(stage);
      // fp16: the unit starts `head` bytes into its window; every row of an eligible view is 8-byte aligned
      const unsigned char* src16 = stage + slab_head(preds + (size_t)h * a.ldh + (size_t)(n0 + sub * PT_HALF) * C);
      for (; q < (h + 1) * KC; q += PT_CONV_GROUPS, ra.step(PT_CONV_GROUPS, SA)) {
        const int kc = q - h * KC;
        const int w = q - SA;                                 // the chunk that held this A slot
        if (w >= 0) {
          ok = pt_wait(&doneK[w & (PT_CHUNK_BARS - 1)], (w / PT_CHUNK_BARS) & 1, abort_s);
          ok = __all_sync(CODA_FULL, ok);
          if (!ok) break;
        }
        unsigned char* dst = aslots + (size_t)ra.slot * 2u * a_limb;
        if constexpr (sizeof(T) == 2) {
          uint2 v[PT_HALF / 32][4];                           // 4 x 4 halves = the 16 columns of this chunk
#pragma unroll
          for (int it = 0; it < PT_HALF / 32; ++it) {
            const unsigned char* rowp = src16 + ((size_t)(it * 32 + lane) * C + kc * 16) * 2u;
#pragma unroll
            for (int j = 0; j < 4; ++j)
              v[it][j] = (kc * 16 + j * 4 < C) ? *reinterpret_cast<const uint2*>(rowp + j * 8) : make_uint2(0u, 0u);
          }
#pragma unroll
          for (int it = 0; it < PT_HALF / 32; ++it) {
            const int item = sub * PT_HALF + it * 32 + lane;
#pragma unroll
            for (int kcore = 0; kcore < 2; ++kcore) {
              const uint2 x = v[it][2 * kcore], y = v[it][2 * kcore + 1];
              const uint32_t off = (uint32_t)((kcore * (PT_M / 8) + (item >> 3)) * 128 + (item & 7) * 16);
              *reinterpret_cast<uint4*>(dst + off) = make_uint4(x.x, x.y, y.x, y.y);
            }
          }
        } else {
        // all loads first: the limb stores below go to shared memory too, so the compiler would not hoist loads over them
        float4 v[PT_HALF / 32][2][2];
#pragma unroll
        for (int it = 0; it < PT_HALF / 32; ++it) {
          const float* rowp = src + (size_t)(it * 32 + lane) * C + kc * 16;
#pragma unroll
          for (int j = 0; j < 4; ++j)                         // 4 x float4 = the 16 columns of this chunk
            v[it][j >> 1][j & 1] = (kc * 16 + j * 4 < C) ? *reinterpret_cast<const float4*>(rowp + j * 4)
                                                          : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int it = 0; it < PT_HALF / 32; ++it) {
          const int item = sub * PT_HALF + it * 32 + lane;
#pragma unroll
          for (int kcore = 0; kcore < 2; ++kcore) {
            const float4 x = v[it][kcore][0], y = v[it][kcore][1];
            uint4 hi, lo;
            pt_split2(x.x, x.y, hi.x, lo.x);
            pt_split2(x.z, x.w, hi.y, lo.y);
            pt_split2(y.x, y.y, hi.z, lo.z);
            pt_split2(y.z, y.w, hi.w, lo.w);
            const uint32_t off = (uint32_t)((kcore * (PT_M / 8) + (item >> 3)) * 128 + (item & 7) * 16);
            *reinterpret_cast<uint4*>(dst + off) = hi;
            *reinterpret_cast<uint4*>(dst + a_limb + off) = lo;
          }
        }
        }
        pt_fence_proxy_async();
        __syncwarp();
        if (lane == 0) pt_arrive(&fullK[q & (PT_CHUNK_BARS - 1)]);
      }
      __syncwarp();
      if (lane == 0) pt_arrive(&emptyS[rs.slot]);
    }
  }

  pt_fence_before();
  __syncthreads();
  if (tid == 0 && *abort_s) atomicOr(a.flags, CODA_B200_FLAG_PIPELINE_TIMEOUT);
  if (warp == 3) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512u) : "memory");
  }
}

struct PiTcPlan {
  int stages, aslots, dslots;
  size_t smem;
};

// shared-memory split: a short ring of converted A chunks, the rest shared between slab staging and D chunks in flight
PiTcPlan pi_tc_plan(int C, int Np, size_t esize) {
  const size_t budget = 227 * 1024;
  const size_t stage = ((size_t)PT_HALF * C * esize + (esize == 4 ? 0 : 16) + 127) & ~(size_t)127;
  const size_t aslot = 2 * (size_t)PT_M * 32, dslot = 2 * (size_t)Np * 32;
  const size_t fixed = (size_t)PT_NBAR * 8 + 64;
  PiTcPlan p;
  p.aslots = PT_CONV_GROUPS + 1;
  p.stages = PT_WARPS_PER_CHUNK + 1;
  p.dslots = 2;
  for (;;) {      // grow the two rings in turn, balancing the BYTES IN FLIGHT (units not being converted, D chunks not being read)
    const size_t used = fixed + p.aslots * aslot + p.stages * stage + p.dslots * dslot;
    const bool more_stage = p.stages < PT_MAX_STAGES && used + stage <= budget;
    const bool more_d = p.dslots < PT_MAX_DSLOTS && used + dslot <= budget;
    if (more_d && ((p.dslots - 1) * dslot <= (p.stages - PT_WARPS_PER_CHUNK) * stage || !more_stage)) ++p.dslots;
    else if (more_stage) ++p.stages;
    else break;
  }
  p.smem = fixed + p.aslots * aslot + p.stages * stage + p.dslots * dslot;
  return p;
}

}  // namespace

extern "C" int coda_b200_pi_full_tc_ok(int H, int64_t N, int C, int64_t model_stride) {
  return H >= 1 && N >= 1 && C >= 16 && C <= 128 && C % 4 == 0 && model_stride % 4 == 0;
}

// the tensor-core and SIMT passes round differently: an fp16 slab is eligible exactly where its fp32 upcast is
extern "C" int coda_b200_pi_full_tc_ok_f16(int H, int64_t N, int C, int64_t model_stride) {
  return coda_b200_pi_full_tc_ok(H, N, C, model_stride);
}

extern "C" size_t coda_b200_pi_full_tc_scratch_bytes(int H, int C) {
  const int Np = (C + 15) / 16 * 16, KC = (C + 15) / 16;
  return (size_t)H * KC * 2 * Np * 16 * 2 + 16;
}

template <typename T>
static int pi_full_tc(const T* preds, int64_t model_stride, const float* D, int H, int64_t N, int C, float* U,
                      void* scratch, uint32_t* flags, coda_stream_t stream) {
  CODA_CHECK_ARG(preds && D && U && scratch && flags, "pi_full_tc: null pointer");
  CODA_CHECK_ARG(coda_b200_pi_full_tc_ok(H, N, C, model_stride),
                 "pi_full_tc: needs 16 <= C <= 128, C %% 4 == 0 and a model stride that is a multiple of 4 (C=%d)", C);
  // fp32: 16-byte aligned copies; fp16: rows 8-byte aligned (the copies take aligned windows)
  CODA_CHECK_ARG(((uintptr_t)preds & (4 * sizeof(T) - 1)) == 0 && ((uintptr_t)U & 15) == 0 && ((uintptr_t)scratch & 15) == 0,
                 "pi_full_tc: preds must be %d-byte aligned, U and scratch 16-byte aligned", (int)(4 * sizeof(T)));
  const int Np = (C + 15) / 16 * 16, KC = (C + 15) / 16;
  unsigned char* wb = reinterpret_cast<unsigned char*>(scratch);
  uint32_t* dmax = reinterpret_cast<uint32_t*>(wb + coda_b200_pi_full_tc_scratch_bytes(H, C) - 16);
  CODA_CUDA_OK(cudaMemsetAsync(dmax, 0, 16, as_stream(stream)));
  k_pi_w_max<<<coda_sm_count(), 256, 0, as_stream(stream)>>>(D, (long long)H * C * C, dmax);
  CODA_LAUNCH_OK("k_pi_w_max");
  k_pi_w_limbs<<<coda_sm_count() * 4, 256, 0, as_stream(stream)>>>(D, H, C, Np, KC, dmax, reinterpret_cast<__half*>(wb));
  CODA_LAUNCH_OK("k_pi_w_limbs");
  const PiTcPlan plan = pi_tc_plan(C, Np, sizeof(T));
  CODA_CHECK_ARG(plan.smem <= 227 * 1024, "pi_full_tc: C=%d does not fit shared memory", C);
  PiTcArgs a;
  a.preds = preds; a.ldh = model_stride; a.wb = wb; a.dmax = dmax; a.U = U; a.flags = flags;
  a.N = N; a.H = H; a.C = C; a.Np = Np; a.KC = KC;
  a.NST = plan.stages; a.SA = plan.aslots; a.SD = plan.dslots;
  // models per drain: the truncating fp32 accumulate of the tensor core loses up to 2^-24 per K = 8 sub-step of the chain
  const char* genv = getenv("CODA_B200_PI_DRAIN");
  a.G = genv ? max(1, min(16, atoi(genv))) : 4;
  CODA_CUDA_OK(cudaFuncSetAttribute(k_pi_full_tc<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)plan.smem));
  const long long grid = (N + PT_M - 1) / PT_M;
  k_pi_full_tc<T><<<(unsigned)grid, PT_THREADS, plan.smem, as_stream(stream)>>>(a);
  CODA_LAUNCH_OK("k_pi_full_tc");
  return CODA_B200_OK;
}

extern "C" int coda_b200_pi_full_tc(const float* preds, int64_t model_stride, const float* D, int H, int64_t N, int C,
                                    float* U, void* scratch, uint32_t* flags, coda_stream_t stream) {
  return pi_full_tc(preds, model_stride, D, H, N, C, U, scratch, flags, stream);
}

extern "C" int coda_b200_pi_full_tc_f16(const uint16_t* preds, int64_t model_stride, const float* D, int H, int64_t N,
                                        int C, float* U, void* scratch, uint32_t* flags, coda_stream_t stream) {
  return pi_full_tc(reinterpret_cast<const __half*>(preds), model_stride, D, H, N, C, U, scratch, flags, stream);
}
