// Slab-streaming kernels of the CODA hot path (HBM-bound passes over the (H, N, C) prediction slab, fp32 or fp16,
// always computed in fp32) and the Bayesian posterior update.
//
//   scan_slab          reference coda.py:193-194 (ensemble mean -> pseudo labels),
//                      coda.py:217-218, 263, 316 (per-model argmax), coda.py:215-219 (unanimity)
//   confusion_accum    coda.py:42   (einsum 'nc,hnj->hcj' with one-hot pseudo labels)
//   init_dirichlets    coda.py:43, 46-63, 196
//   pi_full            coda.py:227-229 (einsum 'hcs,hns->hnc' summed over h, never materialised)
//   pi_reduce          coda.py:230-233
//   label_row / label_apply / pi_rank1   coda.py:316-319 (posterior update + marginal refresh,
//                      restated as the rank-1 column update it algebraically is)
#include "common.cuh"
#include "terms.cuh"

#include <stdlib.h>

// ---------------------------------------------------------------------------------------
// scan_slab: one pass over the slab.  CTA = tile of TN points, all H models.
// ---------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) k_scan_slab(const T* __restrict__ preds, long long ldh, int H, long long N, int C,
                                                   int TN, uint16_t* __restrict__ hard,
                                                   int32_t* __restrict__ pseudo, uint8_t* __restrict__ disagree,
                                                   float* __restrict__ ens_out, uint32_t* __restrict__ flags) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* ens = reinterpret_cast<float*>(smem_raw);                       // [TN][C]
  uint16_t* hard_t = reinterpret_cast<uint16_t*>(ens + (size_t)TN * C);  // [TN][H]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = blockDim.x >> 5;
  const long long n0 = (long long)blockIdx.x * TN;
  const int tn = (int)min((long long)TN, N - n0);
  for (int i = threadIdx.x; i < TN * C; i += blockDim.x) ens[i] = 0.f;
  __syncthreads();
  uint32_t bad = 0;
  for (int h = 0; h < H; ++h) {
    const T* base = preds + (size_t)h * ldh + (size_t)n0 * C;
    for (int p = warp; p < tn; p += nwarp) {
      const T* row = base + (size_t)p * C;
      float* erow = ens + (size_t)p * C;
      float bv = -INFINITY;
      int bi = 0x7fffffff;
      for (int c = lane; c < C; c += 32) {
        float v = slab_ld(row + c);
        if (!isfinite(v)) bad |= CODA_B200_FLAG_NONFINITE_INPUT;
        if (v < 0.f || v > 1.0001f) bad |= CODA_B200_FLAG_RANGE_INPUT;
        erow[c] += v;
        if (v > bv) { bv = v; bi = c; }
      }
      warp_argmax(bv, bi);
      if (lane == 0) hard_t[(size_t)p * H + h] = (uint16_t)(bi == 0x7fffffff ? 0 : bi);
    }
  }
  __syncthreads();
  // hard predictions: contiguous [tn][H] block
  {
    uint16_t* dst = hard + (size_t)n0 * H;
    for (int i = threadIdx.x; i < tn * H; i += blockDim.x) dst[i] = hard_t[i];
  }
  if (ens_out) {   // E[n][c] = sum_h preds[h][n][c], reused by pi_rank1's ensemble shortcut
    float* dst = ens_out + (size_t)n0 * C;
    for (int i = threadIdx.x; i < tn * C; i += blockDim.x) dst[i] = ens[i];
  }
  const float fH = (float)H;
  for (int p = warp; p < tn; p += nwarp) {
    const float* erow = ens + (size_t)p * C;
    float bv = -INFINITY;
    int bi = 0x7fffffff;
    for (int c = lane; c < C; c += 32) {
      float v = erow[c] / fH;   // util.py:14 mean(dim=0), then coda.py:194 argmax
      if (v > bv) { bv = v; bi = c; }
    }
    warp_argmax(bv, bi);
    const uint16_t* hr = hard_t + (size_t)p * H;
    const uint16_t h0 = hr[0];
    int diff = 0;
    for (int h = lane; h < H; h += 32) diff |= (hr[h] != h0);
    diff = __any_sync(CODA_FULL, diff);
    if (lane == 0) {
      pseudo[n0 + p] = (bi == 0x7fffffff ? 0 : bi);
      disagree[n0 + p] = (uint8_t)(diff ? 1 : 0);
    }
  }
  if (bad) atomicOr(flags, bad);
}

// Fast path (C <= 128, N*C % 4 == 0): the [TN x C] tile of every model is one contiguous blob, staged into
// shared memory by 1-D bulk TMA (cp.async.bulk + mbarrier) through a SS_ST-deep ring, so HBM reads run ahead
// of the arg-max / ensemble arithmetic.  Each warp owns 4 rows of the tile (ILP over the four shuffle chains);
// the ensemble sums live in registers.
#define SS_TN 32
#define SS_ST 4
template <typename T, int KC>
__global__ void __launch_bounds__(256) k_scan_slab_tma(const T* __restrict__ preds, long long ldh, int H, long long N, int C,
                                                       uint16_t* __restrict__ hard, int32_t* __restrict__ pseudo,
                                                       uint8_t* __restrict__ disagree, float* __restrict__ ens_out,
                                                       uint32_t* __restrict__ flags) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int tile_floats = SS_TN * C;
  const size_t buf_bytes = ((size_t)tile_floats * sizeof(T) + slab_pad<T>() + 127) / 128 * 128;
  unsigned char* bufs = smem_raw;                                                      // [SS_ST][tile]
  uint16_t* hard_t = reinterpret_cast<uint16_t*>(smem_raw + SS_ST * buf_bytes);         // [SS_TN][H]
  uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + SS_ST * buf_bytes + (((size_t)SS_TN * H * 2 + 15) / 16) * 16);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long n0 = (long long)blockIdx.x * SS_TN;
  const int tn = (int)min((long long)SS_TN, N - n0);
  const uint32_t bytes = (uint32_t)tn * C * sizeof(T);  // fp32: a multiple of 16, callers guarantee (tn * C) % 4 == 0
  if (threadIdx.x == 0) {
    for (int s = 0; s < SS_ST; ++s) mbar_init(&full[s], 1);
    mbar_fence_init();
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int s = 0; s < SS_ST && s < H; ++s)
      tma_load_slab(bufs + s * buf_bytes, preds + (size_t)s * ldh + (size_t)n0 * C, bytes, &full[s]);
  }
  float ens[4][KC];
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int k = 0; k < KC; ++k) ens[r][k] = 0.f;
  uint32_t bad = 0;
  for (int h = 0; h < H; ++h) {
    const int s = h % SS_ST;
    mbar_wait(&full[s], (h / SS_ST) & 1);
    const T* buf = reinterpret_cast<const T*>(bufs + s * buf_bytes + slab_head(preds + (size_t)h * ldh + (size_t)n0 * C));
    float bv[4];
    int bi[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int p = warp + 8 * r;
      bv[r] = -INFINITY;
      bi[r] = 0x7fffffff;
      if (p < tn) {
#pragma unroll
        for (int k = 0; k < KC; ++k) {
          const int c = lane + 32 * k;
          if (c < C) {
            const float v = slab_f(buf[p * C + c]);
            if (!isfinite(v)) bad |= CODA_B200_FLAG_NONFINITE_INPUT;
            if (v < 0.f || v > 1.0001f) bad |= CODA_B200_FLAG_RANGE_INPUT;
            ens[r][k] += v;
            if (v > bv[r]) { bv[r] = v; bi[r] = c; }
          }
        }
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const float ov = __shfl_xor_sync(CODA_FULL, bv[r], o);
        const int oi = __shfl_xor_sync(CODA_FULL, bi[r], o);
        if (ov > bv[r] || (ov == bv[r] && oi < bi[r])) { bv[r] = ov; bi[r] = oi; }
      }
    }
    if (lane == 0) {
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int p = warp + 8 * r;
        if (p < tn) hard_t[(size_t)p * H + h] = (uint16_t)(bi[r] == 0x7fffffff ? 0 : bi[r]);
      }
    }
    __syncthreads();                                   // everyone is done with buf[s]
    if (threadIdx.x == 0 && h + SS_ST < H)
      tma_load_slab(bufs + s * buf_bytes, preds + (size_t)(h + SS_ST) * ldh + (size_t)n0 * C, bytes, &full[s]);
  }
  {
    uint16_t* dst = hard + (size_t)n0 * H;
    for (int i = threadIdx.x; i < tn * H; i += blockDim.x) dst[i] = hard_t[i];
  }
  const float fH = (float)H;
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int p = warp + 8 * r;
    if (p >= tn) continue;
    float bv = -INFINITY;
    int bi = 0x7fffffff;
#pragma unroll
    for (int k = 0; k < KC; ++k) {
      const int c = lane + 32 * k;
      if (c < C) {
        if (ens_out) ens_out[(size_t)(n0 + p) * C + c] = ens[r][k];
        const float v = ens[r][k] / fH;              // util.py:14 mean(dim=0), then coda.py:194 argmax
        if (v > bv) { bv = v; bi = c; }
      }
    }
    warp_argmax(bv, bi);
    const uint16_t* hr = hard_t + (size_t)p * H;
    const uint16_t h0 = hr[0];
    int diff = 0;
    for (int h = lane; h < H; h += 32) diff |= (hr[h] != h0);
    diff = __any_sync(CODA_FULL, diff);
    if (lane == 0) {
      pseudo[n0 + p] = (bi == 0x7fffffff ? 0 : bi);
      disagree[n0 + p] = (uint8_t)(diff ? 1 : 0);
    }
  }
  if (bad) atomicOr(flags, bad);
}

template <typename T>
static int scan_slab(const T* preds, int64_t model_stride, int H, int64_t N, int C, uint16_t* hard, int32_t* pseudo,
                     uint8_t* disagree, float* ens_out, uint32_t* flags, coda_stream_t stream) {
  CODA_CHECK_ARG(preds && hard && pseudo && disagree && flags, "scan_slab: null pointer");
  CODA_CHECK_ARG(model_stride >= (int64_t)N * C, "scan_slab: model_stride %lld < N*C", (long long)model_stride);
  const long long ldh = model_stride;
  CODA_CHECK_ARG(H >= 1 && C >= 2 && C <= 65535 && N >= 1, "scan_slab: bad dims H=%d N=%lld C=%d", H, (long long)N, C);
  // bulk-TMA path when every copy of an fp32 slab is 16-byte aligned.  A 16-bit slab takes it for the same shapes and
  // views (element offsets that are multiples of 4: an 8-byte aligned pointer) and copies aligned windows.
  if (C <= 128 && ldh % 4 == 0 && ((long long)SS_TN * C) % 4 == 0 && ((N % SS_TN) * C) % 4 == 0 &&
      (reinterpret_cast<uintptr_t>(preds) & (4 * sizeof(T) - 1)) == 0) {
    const size_t buf_bytes = ((size_t)SS_TN * C * sizeof(T) + slab_pad<T>() + 127) / 128 * 128;
    const size_t smem = SS_ST * buf_bytes + (((size_t)SS_TN * H * 2 + 15) / 16) * 16 + SS_ST * 8;
    if (smem <= 200 * 1024) {
      const long long grid = (N + SS_TN - 1) / SS_TN;
      cudaStream_t st = as_stream(stream);
#define LAUNCH_SS(KC)                                                                                             \
  do {                                                                                                            \
    CODA_CUDA_OK(cudaFuncSetAttribute(k_scan_slab_tma<T, KC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    k_scan_slab_tma<T, KC><<<(unsigned)grid, 256, smem, st>>>(preds, ldh, H, N, C, hard, pseudo, disagree, ens_out, flags); \
  } while (0)
      if (C <= 32) LAUNCH_SS(1);
      else if (C <= 64) LAUNCH_SS(2);
      else if (C <= 96) LAUNCH_SS(3);
      else LAUNCH_SS(4);
#undef LAUNCH_SS
      CODA_LAUNCH_OK("k_scan_slab_tma");
      return CODA_B200_OK;
    }
  }
  int TN = 32;
  size_t need;
  while (true) {
    need = (size_t)TN * C * 4 + (size_t)TN * H * 2;
    if (need <= 200 * 1024 || TN == 1) break;
    TN >>= 1;
  }
  CODA_CHECK_ARG(need <= 200 * 1024, "scan_slab: H=%d C=%d does not fit shared memory", H, C);
  CODA_CUDA_OK(cudaFuncSetAttribute(k_scan_slab<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)need));
  long long grid = (N + TN - 1) / TN;
  k_scan_slab<T><<<(unsigned)grid, 256, need, as_stream(stream)>>>(preds, ldh, H, N, C, TN, hard, pseudo, disagree, ens_out, flags);
  CODA_LAUNCH_OK("k_scan_slab");
  return CODA_B200_OK;
}

extern "C" int coda_b200_scan_slab(const float* preds, int64_t model_stride, int H, int64_t N, int C, uint16_t* hard,
                                   int32_t* pseudo, uint8_t* disagree, float* ens_out, uint32_t* flags,
                                   coda_stream_t stream) {
  return scan_slab(preds, model_stride, H, N, C, hard, pseudo, disagree, ens_out, flags, stream);
}

extern "C" int coda_b200_scan_slab_f16(const uint16_t* preds, int64_t model_stride, int H, int64_t N, int C,
                                       uint16_t* hard, int32_t* pseudo, uint8_t* disagree, float* ens_out,
                                       uint32_t* flags, coda_stream_t stream) {
  return scan_slab(reinterpret_cast<const __half*>(preds), model_stride, H, N, C, hard, pseudo, disagree, ens_out, flags,
                   stream);
}

// ---------------------------------------------------------------------------------------
// confusion_accum: conf_fx[h][pseudo_n][j] += fx(preds[h][n][j]); int64 fixed point so the
// result does not depend on summation order or on how N is sharded across GPUs.
// grid = (chunks, H).  Shared-memory table when C*C*8 fits, global atomics otherwise.
// ---------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) k_confusion_accum(const T* __restrict__ preds, long long ldh,
                                                         const int32_t* __restrict__ pseudo, int H, long long N,
                                                         int C, float fxs, long long chunk, int use_smem,
                                                         unsigned long long* __restrict__ conf_fx) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  unsigned long long* tab = reinterpret_cast<unsigned long long*>(smem_raw);  // [C][C]
  const int h = blockIdx.y;
  const long long n_lo = (long long)blockIdx.x * chunk;
  const long long n_hi = min(N, n_lo + chunk);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = blockDim.x >> 5;
  unsigned long long* gtab = conf_fx + (size_t)h * C * C;
  if (use_smem) {
    for (int i = threadIdx.x; i < C * C; i += blockDim.x) tab[i] = 0ull;
    __syncthreads();
  }
  unsigned long long* dst_tab = use_smem ? tab : gtab;
  for (long long n = n_lo + warp; n < n_hi; n += nwarp) {
    const int y = pseudo[n];
    const T* row = preds + (size_t)h * ldh + (size_t)n * C;
    unsigned long long* dst = dst_tab + (size_t)y * C;
    for (int j = lane; j < C; j += 32) {
      long long v = to_fx(slab_ld(row + j), fxs);
      if (v != 0) atomicAdd(dst + j, (unsigned long long)v);
    }
  }
  if (use_smem) {
    __syncthreads();
    for (int i = threadIdx.x; i < C * C; i += blockDim.x) {
      unsigned long long v = tab[i];
      if (v) atomicAdd(gtab + i, v);
    }
  }
}

// Class-sorted variant: `order` lists the items grouped by pseudo label, so one warp walks a run of items,
// keeps the int64 column sums of the current class in registers (lane <-> column j) and flushes them with a
// handful of global atomics when the class changes -- no shared-memory atomics on the slab-sized stream.
#define CS_RUN 256
template <typename T, int KC>
__global__ void __launch_bounds__(256) k_confusion_sorted(const T* __restrict__ preds, long long ldh,
                                                          const int32_t* __restrict__ pseudo,
                                                          const int32_t* __restrict__ order, int H, long long N, int C,
                                                          float fxs, unsigned long long* __restrict__ conf_fx) {
  const int h = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long i0 = ((long long)blockIdx.x * 8 + warp) * CS_RUN;
  const long long i1 = min(N, i0 + CS_RUN);
  if (i0 >= N) return;
  const T* slab = preds + (size_t)h * ldh;
  unsigned long long* tab = conf_fx + (size_t)h * C * C;
  long long acc[KC];
#pragma unroll
  for (int k = 0; k < KC; ++k) acc[k] = 0;
  int cur = -1;
  auto flush = [&]() {
    if (cur < 0) return;
#pragma unroll
    for (int k = 0; k < KC; ++k) {
      const int j = lane + 32 * k;
      if (j < C && acc[k]) atomicAdd(tab + (size_t)cur * C + j, (unsigned long long)acc[k]);
      acc[k] = 0;
    }
  };
  for (long long i = i0; i < i1; i += 4) {
    int n[4], y[4];
    float v[4][KC];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const long long ii = min(i + q, i1 - 1);
      n[q] = order[ii];
      y[q] = pseudo[n[q]];
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const T* row = slab + (size_t)n[q] * C;
#pragma unroll
      for (int k = 0; k < KC; ++k) {
        const int j = lane + 32 * k;
        v[q][k] = j < C ? slab_ld(row + j) : 0.f;
      }
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      if (i + q >= i1) break;
      if (y[q] != cur) {
        flush();
        cur = y[q];
      }
#pragma unroll
      for (int k = 0; k < KC; ++k) acc[k] += to_fx(v[q][k], fxs);
    }
  }
  flush();
}

template <typename T>
static int confusion_sorted(const T* preds, int64_t model_stride, const int32_t* pseudo, const int32_t* order, int H,
                            int64_t N, int C, int fx_shift, int64_t* conf_fx, coda_stream_t stream) {
  const long long ldh = model_stride;
  CODA_CHECK_ARG(preds && pseudo && order && conf_fx, "confusion_sorted: null pointer");
  CODA_CHECK_ARG(fx_shift >= 8 && fx_shift <= 46, "confusion_sorted: bad fx_shift %d", fx_shift);
  CODA_CHECK_ARG(C <= 128, "confusion_sorted: C=%d > 128 (use confusion_accum)", C);
  const long long runs = (N + CS_RUN - 1) / CS_RUN;
  dim3 grid((unsigned)((runs + 7) / 8), (unsigned)H);
  const float fxs = exp2f((float)fx_shift);
  unsigned long long* out = reinterpret_cast<unsigned long long*>(conf_fx);
  cudaStream_t st = as_stream(stream);
  if (C <= 32) k_confusion_sorted<T, 1><<<grid, 256, 0, st>>>(preds, ldh, pseudo, order, H, N, C, fxs, out);
  else if (C <= 64) k_confusion_sorted<T, 2><<<grid, 256, 0, st>>>(preds, ldh, pseudo, order, H, N, C, fxs, out);
  else if (C <= 96) k_confusion_sorted<T, 3><<<grid, 256, 0, st>>>(preds, ldh, pseudo, order, H, N, C, fxs, out);
  else k_confusion_sorted<T, 4><<<grid, 256, 0, st>>>(preds, ldh, pseudo, order, H, N, C, fxs, out);
  CODA_LAUNCH_OK("k_confusion_sorted");
  return CODA_B200_OK;
}

extern "C" int coda_b200_confusion_sorted(const float* preds, int64_t model_stride, const int32_t* pseudo,
                                          const int32_t* order, int H, int64_t N, int C, int fx_shift,
                                          int64_t* conf_fx, coda_stream_t stream) {
  return confusion_sorted(preds, model_stride, pseudo, order, H, N, C, fx_shift, conf_fx, stream);
}

extern "C" int coda_b200_confusion_sorted_f16(const uint16_t* preds, int64_t model_stride, const int32_t* pseudo,
                                              const int32_t* order, int H, int64_t N, int C, int fx_shift,
                                              int64_t* conf_fx, coda_stream_t stream) {
  return confusion_sorted(reinterpret_cast<const __half*>(preds), model_stride, pseudo, order, H, N, C, fx_shift, conf_fx,
                          stream);
}

template <typename T>
static int confusion_accum(const T* preds, int64_t model_stride, const int32_t* pseudo, int H, int64_t N, int C,
                           int fx_shift, int64_t* conf_fx, coda_stream_t stream) {
  CODA_CHECK_ARG(preds && pseudo && conf_fx, "confusion_accum: null pointer");
  CODA_CHECK_ARG(fx_shift >= 8 && fx_shift <= 46, "confusion_accum: bad fx_shift %d", fx_shift);
  size_t tab = (size_t)C * C * 8;
  int use_smem = tab <= 160 * 1024;
  size_t smem = use_smem ? tab : 0;
  if (use_smem) CODA_CUDA_OK(cudaFuncSetAttribute(k_confusion_accum<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  long long chunk = 8192;
  long long chunks = (N + chunk - 1) / chunk;
  dim3 grid((unsigned)chunks, (unsigned)H);
  k_confusion_accum<T><<<grid, 256, smem, as_stream(stream)>>>(preds, (long long)model_stride, pseudo, H, N, C, exp2f((float)fx_shift), chunk, use_smem,
                                                           reinterpret_cast<unsigned long long*>(conf_fx));
  CODA_LAUNCH_OK("k_confusion_accum");
  return CODA_B200_OK;
}

extern "C" int coda_b200_confusion_accum(const float* preds, int64_t model_stride, const int32_t* pseudo, int H,
                                         int64_t N, int C, int fx_shift, int64_t* conf_fx, coda_stream_t stream) {
  return confusion_accum(preds, model_stride, pseudo, H, N, C, fx_shift, conf_fx, stream);
}

extern "C" int coda_b200_confusion_accum_f16(const uint16_t* preds, int64_t model_stride, const int32_t* pseudo, int H,
                                             int64_t N, int C, int fx_shift, int64_t* conf_fx, coda_stream_t stream) {
  return confusion_accum(reinterpret_cast<const __half*>(preds), model_stride, pseudo, H, N, C, fx_shift, conf_fx, stream);
}

// ---------------------------------------------------------------------------------------
// init_dirichlets: D = multiplier * (base + prior_strength * conf / max(rowsum, 1e-6))
// one warp per (h, c) row.
// ---------------------------------------------------------------------------------------
__global__ void k_init_dirichlets(const long long* __restrict__ conf_fx, const long long* __restrict__ conf_rest,
                                  int H, int C, int shift,
                                  float prior_strength, float multiplier, int uniform_prior,
                                  float* __restrict__ D) {
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= (long long)H * C) return;
  const int c = (int)(row % C);
  const long long* src = conf_fx + row * C;
  const long long rest = conf_rest ? conf_rest[row] : 0;          // compact slab: carried by every column of the row
  float rs = 0.f;
  for (int j = lane; j < C; j += 32) rs += (float)from_fx(src[j] + rest, shift);
  rs = warp_sum(rs);
  rs = fmaxf(rs, 1e-6f);                                        // coda.py:43 clamp_min(1e-6)
  const float off = uniform_prior ? (float)(2.0 / C) : (float)(1.0 / (C - 1));   // coda.py:53, 57
  for (int j = lane; j < C; j += 32) {
    float conf = (float)from_fx(src[j] + rest, shift) / rs;
    float base = (!uniform_prior && j == c) ? 1.0f : off;       // coda.py:60 fill_diagonal_(1.0)
    D[row * C + j] = multiplier * (base + prior_strength * conf);  // coda.py:63, 196
  }
}

extern "C" int coda_b200_init_dirichlets(const int64_t* conf_fx, const int64_t* conf_rest, int H, int C, int fx_shift,
                                         double prior_strength, double multiplier, int uniform_prior, float* D,
                                         coda_stream_t stream) {
  CODA_CHECK_ARG(conf_fx && D, "init_dirichlets: null pointer");
  long long rows = (long long)H * C;
  int wpb = 8;
  k_init_dirichlets<<<(unsigned)((rows + wpb - 1) / wpb), wpb * 32, 0, as_stream(stream)>>>(
      reinterpret_cast<const long long*>(conf_fx), reinterpret_cast<const long long*>(conf_rest), H, C, fx_shift,
      (float)prior_strength, (float)multiplier,
      uniform_prior, D);
  CODA_LAUNCH_OK("k_init_dirichlets");
  return CODA_B200_OK;
}

// ---------------------------------------------------------------------------------------
// pi_full: U[n][c] = sum_h sum_s D[h][c][s] * preds[h][n][s]   (fp32 SIMT GEMM, K = H*C)
// CTA: 64 points x (up to 128 classes per pass); thread (pg, cg) owns 4 points x 8 classes.
// ---------------------------------------------------------------------------------------
#define PF_TN 64
#define PF_TC 128
#define PF_SK 32
template <typename T>
__global__ void __launch_bounds__(256) k_pi_full(const T* __restrict__ preds, long long ldh,
                                                 const float* __restrict__ D, int H, long long N, int C,
                                                 float* __restrict__ U) {
  __shared__ float As[PF_TN][PF_SK + 1];
  __shared__ float Bs[PF_TC][PF_SK + 1];
  const int tid = threadIdx.x;
  const int pg = tid >> 4, cg = tid & 15;
  const long long n0 = (long long)blockIdx.x * PF_TN;
  for (int c0 = 0; c0 < C; c0 += PF_TC) {
    float acc[4][8];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int k = 0; k < 8; ++k) acc[i][k] = 0.f;
    for (int h = 0; h < H; ++h) {
      const T* Ah = preds + (size_t)h * ldh;
      const float* Dh = D + ((size_t)h * C) * C;
      for (int s0 = 0; s0 < C; s0 += PF_SK) {
        __syncthreads();
        for (int e = tid; e < PF_TN * PF_SK; e += 256) {
          int r = e >> 5, col = e & 31;
          long long n = n0 + r;
          int s = s0 + col;
          As[r][col] = (n < N && s < C) ? slab_ld(Ah + (size_t)n * C + s) : 0.f;
        }
        for (int e = tid; e < PF_TC * PF_SK; e += 256) {
          int r = e >> 5, col = e & 31;
          int c = c0 + r, s = s0 + col;
          Bs[r][col] = (c < C && s < C) ? __ldg(Dh + (size_t)c * C + s) : 0.f;
        }
        __syncthreads();
#pragma unroll 8
        for (int s = 0; s < PF_SK; ++s) {
          float a[4], b[8];
#pragma unroll
          for (int i = 0; i < 4; ++i) a[i] = As[pg * 4 + i][s];
#pragma unroll
          for (int k = 0; k < 8; ++k) b[k] = Bs[cg + 16 * k][s];
#pragma unroll
          for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int k = 0; k < 8; ++k) acc[i][k] = fmaf(a[i], b[k], acc[i][k]);
        }
      }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      long long n = n0 + pg * 4 + i;
      if (n >= N) continue;
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        int c = c0 + cg + 16 * k;
        if (c < C) U[(size_t)n * C + c] = acc[i][k];
      }
    }
  }
}

template <typename T>
static int pi_full(const T* preds, int64_t model_stride, const float* D, int H, int64_t N, int C, float* U,
                   coda_stream_t stream) {
  CODA_CHECK_ARG(preds && D && U, "pi_full: null pointer");
  long long grid = (N + PF_TN - 1) / PF_TN;
  k_pi_full<T><<<(unsigned)grid, 256, 0, as_stream(stream)>>>(preds, (long long)model_stride, D, H, N, C, U);
  CODA_LAUNCH_OK("k_pi_full");
  return CODA_B200_OK;
}

extern "C" int coda_b200_pi_full(const float* preds, int64_t model_stride, const float* D, int H, int64_t N, int C,
                                 float* U, coda_stream_t stream) {
  return pi_full(preds, model_stride, D, H, N, C, U, stream);
}

extern "C" int coda_b200_pi_full_f16(const uint16_t* preds, int64_t model_stride, const float* D, int H, int64_t N, int C,
                                     float* U, coda_stream_t stream) {
  return pi_full(reinterpret_cast<const __half*>(preds), model_stride, D, H, N, C, U, stream);
}

// ---------------------------------------------------------------------------------------
// shared tail of pi_reduce / pi_rank1: one warp normalises one row of U and accumulates the
// per-class column sums of pi_hat_xi (fixed point) into a warp-private shared-memory vector.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ void row_accumulate(float* __restrict__ urow, int C, int lane, float fxs, int t,
                                               float delta_t, float* __restrict__ xi_out,
                                               long long* __restrict__ wacc, uint32_t& bad) {
  float s = 0.f, ut = 0.f;
  for (int c = lane; c < C; c += 32) {      // loads only: a store inside this loop would order every later load behind it
    float u = urow[c];                       // (possible alias) and turn the row into C / 32 dependent round trips
    if (c == t) {
      u += delta_t;
      ut = u;
    }
    s += u;
  }
  if (t >= 0 && lane == (t & 31)) urow[t] = ut;
  s = warp_sum(s);
  if (!isfinite(s)) bad |= CODA_B200_FLAG_NONFINITE_PI;
  const float den = fmaxf(s, 1e-12f);                               // coda.py:230 clamp_(min=1e-12)
  const float rden = 1.0f / den;
  for (int c = lane; c < C; c += 32) {
    float xi = row_quot(urow[c], den, rden);   // column t was rewritten above by this same lane

    if (xi_out) xi_out[c] = xi;
    wacc[c] += to_fx(xi, fxs);
  }
}

__global__ void __launch_bounds__(256) k_pi_reduce(float* __restrict__ U, long long N, int C, float fxs,
                                                   float* __restrict__ xi_out,
                                                   unsigned long long* __restrict__ pisum_fx,
                                                   uint32_t* __restrict__ flags) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  long long* wacc_all = reinterpret_cast<long long*>(smem_raw);       // [nwarp][C]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = blockDim.x >> 5;
  long long* wacc = wacc_all + (size_t)warp * C;
  for (int c = lane; c < C; c += 32) wacc[c] = 0;
  __syncwarp();
  uint32_t bad = 0;
  for (long long n = (long long)blockIdx.x * nwarp + warp; n < N; n += (long long)gridDim.x * nwarp)
    row_accumulate(U + (size_t)n * C, C, lane, fxs, -1, 0.f, xi_out ? xi_out + (size_t)n * C : nullptr, wacc, bad);
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    long long s = 0;
    for (int w = 0; w < nwarp; ++w) s += wacc_all[(size_t)w * C + c];
    if (s) atomicAdd(pisum_fx + c, (unsigned long long)s);
  }
  if (bad) atomicOr(flags, bad);
}

extern "C" int coda_b200_pi_reduce(float* U, int64_t N, int C, int fx_shift, float* xi_out, int64_t* pisum_fx,
                                   uint32_t* flags, coda_stream_t stream) {
  CODA_CHECK_ARG(U && pisum_fx && flags, "pi_reduce: null pointer");
  size_t smem = (size_t)8 * C * 8;
  CODA_CHECK_ARG(smem <= 200 * 1024, "pi_reduce: C=%d too large", C);
  CODA_CUDA_OK(cudaFuncSetAttribute(k_pi_reduce, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  long long want = (N + 7) / 8;
  int grid = (int)min(want, (long long)coda_sm_count() * 8);
  k_pi_reduce<<<grid, 256, smem, as_stream(stream)>>>(U, N, C, exp2f((float)fx_shift), xi_out,
                                                      reinterpret_cast<unsigned long long*>(pisum_fx), flags);
  CODA_LAUNCH_OK("k_pi_reduce");
  return CODA_B200_OK;
}

// ---------------------------------------------------------------------------------------
// posterior update (coda.py:316-317) and the marginal refresh it triggers (coda.py:319),
// restated:  D[h, t, j_h] += lr   with j_h = p_h(idx)   changes only row t of every D[h], so
//   U[n, t] += lr * sum_h preds[h, n, j_h]      and every other column of U is untouched.
// (the label itself -- owner's p_h(idx), labeled mark, D update, gather list -- is in step.cu)
// pi_rank1    : gathers one float per (h, n) (one 32 B sector each), updates column t of U,
//               renormalises rows on the fly and re-accumulates sum_n pi_hat_xi[n, :]
// ---------------------------------------------------------------------------------------
// ---------------------------------------------------------------------------------------
// class-major shadow copy  T[s][c][n] = preds[h_s][n][c]  for a subset of models (as many as spare HBM
// allows, least accurate first).  The rank-1 refresh needs ONE float per (model, item): from the reference
// layout that costs a 64-byte DRAM fetch each, from the shadow it is a coalesced 4-byte read.
// grid = (ceil(N/32), ceil(C/32), S), block = (32, 8)
// ---------------------------------------------------------------------------------------
template <typename E>
__global__ void k_shadow_transpose(const E* __restrict__ preds, long long ldh, long long N, int C,
                                   const int32_t* __restrict__ model_of_slot, long long cs, E* __restrict__ T) {
  __shared__ E tile[32][33];
  const int s = blockIdx.z, h = model_of_slot[s];
  const long long n0 = (long long)blockIdx.x * 32;
  const int c0 = blockIdx.y * 32;
  const E* src = preds + (size_t)h * ldh;
  for (int r = threadIdx.y; r < 32; r += 8) {
    const long long n = n0 + r;
    const int c = c0 + threadIdx.x;
    tile[r][threadIdx.x] = (n < N && c < C) ? __ldg(src + (size_t)n * C + c) : E(0.f);
  }
  __syncthreads();
  E* dst = T + (size_t)s * C * cs;
  for (int r = threadIdx.y; r < 32; r += 8) {
    const int c = c0 + r;
    const long long n = n0 + threadIdx.x;
    if (c < C && n < N) dst[(size_t)c * cs + n] = tile[threadIdx.x][r];
  }
}

template <typename E>
static int shadow_build(const E* preds, int64_t model_stride, int H, int64_t N, int C, const int32_t* model_of_slot, int S,
                        int64_t col_stride, E* T, coda_stream_t stream) {
  CODA_CHECK_ARG(preds && model_of_slot && T && S >= 1 && S <= H && col_stride >= N, "shadow_build: bad arguments");
  CODA_CHECK_ARG(sizeof(E) == 4 || col_stride % 8 == 0, "shadow_build: col_stride %lld leaves fp16 columns unaligned",
                 (long long)col_stride);
  long long gx = (N + 31) / 32;
  CODA_CHECK_ARG(gx <= 0x7fffffffLL && S <= 65535, "shadow_build: grid too large");
  dim3 grid((unsigned)gx, (unsigned)((C + 31) / 32), (unsigned)S), block(32, 8);
  k_shadow_transpose<E><<<grid, block, 0, as_stream(stream)>>>(preds, (long long)model_stride, N, C, model_of_slot,
                                                               (long long)col_stride, T);
  CODA_LAUNCH_OK("k_shadow_transpose");
  return CODA_B200_OK;
}

extern "C" int coda_b200_shadow_build(const float* preds, int64_t model_stride, int H, int64_t N, int C,
                                      const int32_t* model_of_slot, int S, int64_t col_stride, float* T,
                                      coda_stream_t stream) {
  return shadow_build(preds, model_stride, H, N, C, model_of_slot, S, col_stride, T, stream);
}

extern "C" int coda_b200_shadow_build_f16(const uint16_t* preds, int64_t model_stride, int H, int64_t N, int C,
                                          const int32_t* model_of_slot, int S, int64_t col_stride, uint16_t* T,
                                          coda_stream_t stream) {
  return shadow_build(reinterpret_cast<const __half*>(preds), model_stride, H, N, C, model_of_slot, S, col_stride,
                      reinterpret_cast<__half*>(T), stream);
}

// register variant of row_accumulate for C <= 32 * KC: NR rows per call (all loads issued before the first
// reduction), the int64 column sums stay in registers
template <int KC, int NR>
__device__ __forceinline__ void rows_accumulate_reg(float* __restrict__ U, long long row0, int nrows, int rstride,
                                                    int C, int lane, float fxs, int t, const float (&dv)[NR],
                                                    long long (&racc)[KC], uint32_t& bad) {
  float u[NR][KC];
#pragma unroll
  for (int r = 0; r < NR; ++r) {
    const bool ok = r * rstride < nrows;
    const float* urow = U + (size_t)(row0 + (ok ? r * rstride : 0)) * C;
#pragma unroll
    for (int k = 0; k < KC; ++k) {
      const int c = lane + 32 * k;
      u[r][k] = (ok && c < C) ? urow[c] : 0.f;
    }
  }
#pragma unroll
  for (int r = 0; r < NR; ++r) {
    if (r * rstride >= nrows) break;
    float* urow = U + (size_t)(row0 + r * rstride) * C;
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < KC; ++k) {
      const int c = lane + 32 * k;
      if (c == t) {
        u[r][k] += dv[r];
        urow[c] = u[r][k];
      }
      s += u[r][k];
    }
    s = warp_sum(s);
    if (!isfinite(s)) bad |= CODA_B200_FLAG_NONFINITE_PI;
    const float den = fmaxf(s, 1e-12f);                             // coda.py:230 clamp_(min=1e-12)
    const float rden = 1.0f / den;
#pragma unroll
    for (int k = 0; k < KC; ++k) racc[k] += to_fx(row_quot(u[r][k], den, rden), fxs);
  }
}

// The gather list is read by every lane at the same index: the constant cache serves that as a uniform load, shared
// memory as a broadcast LDS through the MIO pipe (measured: 0.37 ms vs 0.55 ms for the kernel below at cfg3).  The
// constant bank is per device and shared by every stream of the process, so it is cut into slots: a caller that owns
// a slot (coda_b200_pi_rank1's const_slot >= 0; coda_b200.engine hands them out per device) gets the constant path,
// anyone else the shared-memory copy.
#define R1_CONST_TERMS 3584                        // 56 KB of the 64 KB constant bank
__constant__ R1Term c_terms_bank[R1_CONST_TERMS];

#define R1_TN 256
// GU: gathers in flight per lane, NR: U rows in flight per warp (more of both = more bytes in flight per SM at
// the price of registers / resident warps)
template <typename T, int KC, int GU = 16, int NR = 4, bool CONST_TERMS = false>
__global__ void __launch_bounds__(256, (GU > 16 ? 3 : 4)) k_pi_rank1(const T* __restrict__ preds, const float* __restrict__ E,
                                                  long long N, int C, const long long* __restrict__ sel,
                                                  const int32_t* __restrict__ hdr, const R1Term* __restrict__ gterms,
                                                  int const_base, float lr, float fxs,
                                                  float* __restrict__ U, unsigned long long* __restrict__ pisum_fx,
                                                  uint32_t* __restrict__ flags) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  long long* wacc_all = reinterpret_cast<long long*>(smem_raw);                 // [8][C]
  R1Term* s_terms = reinterpret_cast<R1Term*>(wacc_all + (size_t)8 * C);        // [nt] gather list (broadcast reads)
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int t = (int)sel[1];
  const int nt = hdr[0], tp = hdr[1];
  if (!CONST_TERMS)
    for (int k = threadIdx.x; k < nt; k += blockDim.x) s_terms[k] = gterms[k];
  const R1Term* c_terms = CONST_TERMS ? (c_terms_bank + const_base) : s_terms;
  long long* wacc = wacc_all + (size_t)warp * C;
  for (int c = lane; c < C; c += 32) wacc[c] = 0;
  long long racc[KC > 0 ? KC : 1];
#pragma unroll
  for (int k = 0; k < (KC > 0 ? KC : 1); ++k) racc[k] = 0;
  __syncthreads();
  uint32_t bad = 0;
  // one warp = 32 consecutive items: lane i gathers item i's increment, then the warp walks the 32 rows of U
  // (increment handed over by shuffle).  No block-level barrier inside the loop, warps run independently.
  const long long wstride = (long long)gridDim.x * R1_TN;
  for (long long n0 = (long long)blockIdx.x * R1_TN + warp * 32; n0 < N; n0 += wstride) {
    const long long n = n0 + lane;
    float d = 0.f;
    if (n < N) {
      if (tp >= 0) d = __ldg(E + (size_t)n * C + tp);
      int k = 0;
      for (; k + GU <= nt; k += GU) {
        float v[GU];
#pragma unroll
        for (int q = 0; q < GU; ++q) v[q] = slab_ld(preds + c_terms[k + q].off + n * c_terms[k + q].str);
#pragma unroll
        for (int q = 0; q < GU; ++q) d = fmaf(c_terms[k + q].sg, v[q], d);
      }
      for (; k < nt; ++k) d = fmaf(c_terms[k].sg, slab_ld(preds + c_terms[k].off + n * c_terms[k].str), d);
    }
    const float dl = lr * d;
    const int rows = (int)min(32LL, N - n0);
    if (KC > 0) {
      for (int r = 0; r < rows; r += NR) {
        float dv[NR];
#pragma unroll
        for (int i = 0; i < NR; ++i) dv[i] = __shfl_sync(CODA_FULL, dl, (r + i) & 31);
        rows_accumulate_reg<(KC > 0 ? KC : 1), NR>(U, n0 + r, rows - r, 1, C, lane, fxs, t, dv, racc, bad);
      }
    } else {
      for (int r = 0; r < rows; ++r) {
        const float dr = __shfl_sync(CODA_FULL, dl, r);
        row_accumulate(U + (size_t)(n0 + r) * C, C, lane, fxs, t, dr, nullptr, wacc, bad);
      }
    }
  }
  if (KC > 0) {
#pragma unroll
    for (int k = 0; k < (KC > 0 ? KC : 1); ++k) {
      const int c = lane + 32 * k;
      if (c < C) wacc[c] = racc[k];
    }
  }
  __syncthreads();          // every warp's column sums are in shared memory
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    long long s2 = 0;
    for (int w = 0; w < 8; ++w) s2 += wacc_all[(size_t)w * C + c];
    if (s2) atomicAdd(pisum_fx + c, (unsigned long long)s2);
  }
  if (bad) atomicOr(flags, bad);
}

// pi_rank1 with four consecutive items per lane (C <= 128): a warp owns 128 consecutive items, so every gather
// from the class-major shadow is one 512-byte contiguous run per term (float4 per lane) instead of 128 bytes --
// four times fewer DRAM page switches for the same bytes.  Same arithmetic, same order as k_pi_rank1.
#define R1V_WI 128     // items per warp
template <int KC>
__global__ void __launch_bounds__(256, 3) k_pi_rank1_v4(const float* __restrict__ preds, const float* __restrict__ E,
                                                     long long N, int C, const long long* __restrict__ sel,
                                                     const int32_t* __restrict__ hdr, const R1Term* __restrict__ gterms,
                                                     float lr, float fxs, float* __restrict__ U,
                                                     unsigned long long* __restrict__ pisum_fx,
                                                     uint32_t* __restrict__ flags) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  long long* wacc_all = reinterpret_cast<long long*>(smem_raw);                 // [8][C]
  R1Term* c_terms = reinterpret_cast<R1Term*>(wacc_all + (size_t)8 * C);        // [nt]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int t = (int)sel[1];
  const int nt = hdr[0], tp = hdr[1];
  for (int k = threadIdx.x; k < nt; k += blockDim.x) c_terms[k] = gterms[k];
  long long racc[KC];
#pragma unroll
  for (int k = 0; k < KC; ++k) racc[k] = 0;
  __syncthreads();
  uint32_t bad = 0;
  const long long cta_items = (long long)8 * R1V_WI;
  for (long long n0 = (long long)blockIdx.x * cta_items + (long long)warp * R1V_WI; n0 < N; n0 += (long long)gridDim.x * cta_items) {
    const long long nl = n0 + 4 * lane;
    const bool full4 = nl + 3 < N;
    float d[4] = {0.f, 0.f, 0.f, 0.f};
    if (tp >= 0) {
#pragma unroll
      for (int i = 0; i < 4; ++i)
        if (nl + i < N) d[i] = __ldg(E + (size_t)(nl + i) * C + tp);
    }
    int k = 0;
    for (; k + 8 <= nt; k += 8) {
      float v[8][4];
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const R1Term tm = c_terms[k + q];
        if (tm.str == 1 && full4) {
          const float4 x = __ldg(reinterpret_cast<const float4*>(preds + tm.off + nl));
          v[q][0] = x.x; v[q][1] = x.y; v[q][2] = x.z; v[q][3] = x.w;
        } else {
#pragma unroll
          for (int i = 0; i < 4; ++i) v[q][i] = (nl + i < N) ? __ldg(preds + tm.off + (nl + i) * tm.str) : 0.f;
        }
      }
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const float sg = c_terms[k + q].sg;
#pragma unroll
        for (int i = 0; i < 4; ++i) d[i] = fmaf(sg, v[q][i], d[i]);
      }
    }
    for (; k < nt; ++k) {
      const R1Term tm = c_terms[k];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float x = (nl + i < N) ? __ldg(preds + tm.off + (nl + i) * tm.str) : 0.f;
        d[i] = fmaf(tm.sg, x, d[i]);
      }
    }
    float dl[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) dl[i] = lr * d[i];
    const int rows = (int)min((long long)R1V_WI, N - n0);
    for (int r = 0; r < rows; r += 4) {
      float dv[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) dv[i] = __shfl_sync(CODA_FULL, dl[i], r >> 2);
      rows_accumulate_reg<KC, 4>(U, n0 + r, rows - r, 1, C, lane, fxs, t, dv, racc, bad);
    }
  }
  long long* wacc = wacc_all + (size_t)warp * C;
#pragma unroll
  for (int k = 0; k < KC; ++k) {
    const int c = lane + 32 * k;
    if (c < C) wacc[c] = racc[k];
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    long long s2 = 0;
    for (int w = 0; w < 8; ++w) s2 += wacc_all[(size_t)w * C + c];
    if (s2) atomicAdd(pisum_fx + c, (unsigned long long)s2);
  }
  if (bad) atomicOr(flags, bad);
}

// ---------------------------------------------------------------------------------------
// pi_rank1, bulk-TMA pipeline (C <= 128): the same arithmetic in the same order as k_pi_rank1, fed differently.
// A persistent CTA walks tiles of TR items.  Everything a tile needs is contiguous in HBM:
//   * the U rows of the tile            TR*C floats   -> ONE cp.async.bulk into shared memory (warp 9)
//   * per shadow term, the TR increments  TR floats    -> one cp.async.bulk each into a ring of ST stages x TB terms (warp 8)
// so the memory system runs ahead of the arithmetic without holding anything in registers.  Consumer warp w owns
// items [32w, 32w+32) of the tile: lane i sums item i's terms in list order (ring slots by LDS, the few terms of
// models without a shadow slot by a direct gather), then the warp walks its 32 rows of the U tile (increment handed
// over by shuffle), renormalises, accumulates the int64 column sums in registers and stores column t back.
// ---------------------------------------------------------------------------------------
#define R1X_THREADS 320      // 8 consumer warps + ring producer warp + U producer warp
#define R1X_ST 4
#define R1X_TB 16

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

template <int KC>
__global__ void __launch_bounds__(R1X_THREADS, 1) k_pi_rank1_tma(const float* __restrict__ preds,
                                                                 const float* __restrict__ E, long long N, int C, int TR,
                                                                 const long long* __restrict__ sel,
                                                                 const int32_t* __restrict__ hdr,
                                                                 const R1Term* __restrict__ gterms, float lr, float fxs,
                                                                 float* __restrict__ U,
                                                                 unsigned long long* __restrict__ pisum_fx,
                                                                 uint32_t* __restrict__ flags) {
  extern __shared__ __align__(128) unsigned char smem_r1x[];
  unsigned char* smem_raw = smem_r1x;
  const int nt = hdr[0], tp = hdr[1];
  const int t = (int)sel[1];
  const size_t u_bytes = ((size_t)TR * C * 4 + 127) & ~(size_t)127;
  float* Ut = reinterpret_cast<float*>(smem_raw);                                        // [TR][C]
  float* ring = reinterpret_cast<float*>(smem_raw + u_bytes);                            // [ST][TB][TR]
  R1Term* terms = reinterpret_cast<R1Term*>(ring + (size_t)R1X_ST * R1X_TB * TR);        // [nt]
  long long* wacc_all = reinterpret_cast<long long*>(terms + nt);                        // [8][C]
  int* shl = reinterpret_cast<int*>(wacc_all + (size_t)8 * C);                           // [nt] indices of the shadow terms
  uint64_t* bars = reinterpret_cast<uint64_t*>((reinterpret_cast<uintptr_t>(shl + nt) + 7) & ~(uintptr_t)7);
  uint64_t* fullU = bars, *emptyU = bars + 1, *full = bars + 2, *empty = bars + 2 + R1X_ST;
  __shared__ int s_nsh;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int nwarp_act = TR >> 5;                                                         // consumer warps with rows
  for (int k = tid; k < nt; k += R1X_THREADS) terms[k] = gterms[k];
  for (int c = tid; c < 8 * C; c += R1X_THREADS) wacc_all[c] = 0;
  if (tid == 0) {
    mbar_init(fullU, 1);
    mbar_init(emptyU, nwarp_act);
    for (int s = 0; s < R1X_ST; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], nwarp_act); }
    mbar_fence_init();
  }
  __syncthreads();
  if (tid == 0) {                               // shadow terms in list order (cheap: nt <= 2H)
    int n = 0;
    for (int k = 0; k < nt; ++k)
      if (terms[k].str == 1) shl[n++] = k;
    s_nsh = n;
  }
  __syncthreads();
  const int nsh = s_nsh;
  const int nch = (nsh + R1X_TB - 1) / R1X_TB;                                            // ring chunks per tile
  const long long ntiles = (N + TR - 1) / TR;

  if (warp == 8) {                              // ---- ring producer ----
    if (lane == 0) {
      long long gch = 0;
      for (long long ti = blockIdx.x; ti < ntiles; ti += gridDim.x) {
        const long long n0 = ti * TR;
        const int rows = (int)min((long long)TR, N - n0);
        const uint32_t rb = (uint32_t)((rows + 3) & ~3) * 4u;                             // columns are padded to 4 items
        for (int c = 0; c < nch; ++c, ++gch) {
          const int s = (int)(gch % R1X_ST);
          if (gch >= R1X_ST) mbar_wait(&empty[s], (uint32_t)(((gch / R1X_ST) - 1) & 1));
          const int cnt = min(R1X_TB, nsh - c * R1X_TB);
          mbar_expect_tx(&full[s], (uint32_t)cnt * rb);
          for (int j = 0; j < cnt; ++j)
            tma_load_1d(ring + ((size_t)s * R1X_TB + j) * TR, preds + terms[shl[c * R1X_TB + j]].off + n0, rb, &full[s]);
        }
      }
    }
    return;
  }
  if (warp == 9) {                              // ---- U tile producer ----
    if (lane == 0) {
      long long it = 0;
      for (long long ti = blockIdx.x; ti < ntiles; ti += gridDim.x, ++it) {
        const long long n0 = ti * TR;
        const int rows = (int)min((long long)TR, N - n0);
        const uint32_t ub = ((uint32_t)rows * C * 4u + 15u) & ~15u;                       // U carries 16 bytes of slack
        if (it > 0) mbar_wait(emptyU, (uint32_t)((it - 1) & 1));
        mbar_expect_tx(fullU, ub);
        tma_load_1d(Ut, U + (size_t)n0 * C, ub, fullU);
      }
    }
    return;
  }
  if (warp >= nwarp_act) return;
  // ---- consumers ----
  long long racc[KC];
#pragma unroll
  for (int k = 0; k < KC; ++k) racc[k] = 0;
  uint32_t bad = 0;
  long long gch = 0, it = 0;
  for (long long ti = blockIdx.x; ti < ntiles; ti += gridDim.x, ++it) {
    const long long n0 = ti * TR;
    const int rows = (int)min((long long)TR, N - n0);
    const int li = warp * 32 + lane;                 // this lane's item within the tile
    const long long n = n0 + li;
    const bool valid = li < rows;
    float d = 0.f;
    if (valid && tp >= 0) d = __ldg(E + (size_t)n * C + tp);
    int shi = 0;                                     // shadow terms consumed in this tile
    const float* slot = ring;
    for (int k = 0; k < nt; ++k) {
      const R1Term tm = terms[k];
      float v = 0.f;
      if (tm.str == 1) {
        const int j = shi % R1X_TB;
        if (j == 0) {
          const long long g = gch + shi / R1X_TB;
          const int s = (int)(g % R1X_ST);
          mbar_wait(&full[s], (uint32_t)((g / R1X_ST) & 1));
          slot = ring + (size_t)s * R1X_TB * TR;
        }
        v = slot[(size_t)j * TR + li];
        ++shi;
        if (j == R1X_TB - 1 || shi == nsh) {         // last read of this stage by this warp
          __syncwarp();
          if (lane == 0) mbar_arrive(&empty[(int)((gch + (shi - 1) / R1X_TB) % R1X_ST)]);
        }
      } else if (valid) {
        v = __ldg(preds + tm.off + n * tm.str);
      }
      d = fmaf(tm.sg, v, d);
    }
    gch += nch;
    const float dl = valid ? lr * d : 0.f;
    // ---- row pass over this warp's 32 rows of the U tile ----
    mbar_wait(fullU, (uint32_t)(it & 1));
    const int wrows = min(32, rows - warp * 32);
    for (int r = 0; r < wrows; r += 4) {
      float u[4][KC], dv[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        dv[i] = __shfl_sync(CODA_FULL, dl, (r + i) & 31);
        const float* urow = Ut + (size_t)(warp * 32 + min(r + i, wrows - 1)) * C;
#pragma unroll
        for (int k = 0; k < KC; ++k) {
          const int c = lane + 32 * k;
          u[i][k] = c < C ? urow[c] : 0.f;
        }
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        if (r + i >= wrows) break;
        float s = 0.f;
#pragma unroll
        for (int k = 0; k < KC; ++k) {
          const int c = lane + 32 * k;
          if (c == t) {
            u[i][k] += dv[i];
            U[(size_t)(n0 + warp * 32 + r + i) * C + c] = u[i][k];
          }
          s += u[i][k];
        }
        s = warp_sum(s);
        if (!isfinite(s)) bad |= CODA_B200_FLAG_NONFINITE_PI;
        const float den = fmaxf(s, 1e-12f);                             // coda.py:230 clamp_(min=1e-12)
        const float rden = 1.0f / den;
#pragma unroll
        for (int k = 0; k < KC; ++k) racc[k] += to_fx(row_quot(u[i][k], den, rden), fxs);
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(emptyU);
  }
  long long* wacc = wacc_all + (size_t)warp * C;
#pragma unroll
  for (int k = 0; k < KC; ++k) {
    const int c = lane + 32 * k;
    if (c < C) wacc[c] = racc[k];
  }
  // consumer-only barrier (the producer warps have left): named barrier 1
  asm volatile("bar.sync 1, %0;" ::"r"(nwarp_act * 32) : "memory");
  for (int c = tid; c < C; c += nwarp_act * 32) {
    long long s2 = 0;
    for (int w = 0; w < nwarp_act; ++w) s2 += wacc_all[(size_t)w * C + c];
    if (s2) atomicAdd(pisum_fx + c, (unsigned long long)s2);
  }
  if (bad) atomicOr(flags, bad);
}

static int r1x_tile_rows(int C) {     // rows per tile: U tile <= ~104 KB, multiple of 32, <= 256
  int tr = (int)((104 * 1024) / ((size_t)C * 4)) / 32 * 32;
  if (tr > 256) tr = 256;
  return tr;
}

template <typename T>
static int pi_rank1(const T* preds, const float* ens, int H, int64_t N, int C, const int64_t* sel, double lr,
                    int fx_shift, const int32_t* terms /*[2 + 8H]*/, float* U, int64_t* pisum_fx, uint32_t* flags,
                    int ctas_per_sm, int const_slot, coda_stream_t stream) {
  CODA_CHECK_ARG(preds && sel && terms && U && pisum_fx && flags, "pi_rank1: null pointer");
  CODA_CHECK_ARG(2 * H <= R1_MAXT, "pi_rank1: H=%d too large", H);
  CODA_CHECK_ARG((reinterpret_cast<uintptr_t>(terms) & 7) == 0, "pi_rank1: terms must be 8-byte aligned");
  const int32_t* hdr = terms;                                                  // 2 ints
  const R1Term* tlist = reinterpret_cast<const R1Term*>(terms + 2);            // <= 2H x 16 bytes
  cudaStream_t st = as_stream(stream);
  // bulk-TMA pipeline: C <= 128, 16-byte aligned U / preds / E, item counts that keep every bulk copy aligned
  // variants (identical bits): "v1" one item per lane (default; measured fastest: 0.40 ms at cfg3), "v4" four items
  // per lane / 512-byte runs per term (0.51 ms), "tma" the bulk-TMA pipeline (1.2 ms: 8 consumer warps per SM in
  // lock-step phases).  CODA_B200_R1 selects one for A/B runs.
  const char* r1env = getenv("CODA_B200_R1");
  const bool want_tma = r1env && r1env[0] == 't';
  const bool want_v1 = !(r1env && r1env[0] == 'v' && r1env[1] == '4');
  const bool want_deep = r1env && r1env[0] == 'v' && r1env[1] == '1' && r1env[2] == 'd';   // "v1d": 32 gathers / 8 rows in flight
  const bool no_tma = !want_tma;
  // the "tma" and "v4" variants read the slab as fp32 words (bulk copies of shadow columns, float4 runs): fp32 only
  CODA_CHECK_ARG(sizeof(T) == 4 || (!want_tma && want_v1),
                 "pi_rank1: CODA_B200_R1=%s is not available for a 16-bit slab (use v1 or v1d)", r1env ? r1env : "");
  const int TR = C <= 128 ? r1x_tile_rows(C) : 0;
  if constexpr (sizeof(T) == 4) if (!no_tma && TR >= 32 && (reinterpret_cast<uintptr_t>(U) & 15) == 0) {
    const size_t u_bytes = ((size_t)TR * C * 4 + 127) & ~(size_t)127;
    const size_t smem_x = u_bytes + (size_t)R1X_ST * R1X_TB * TR * 4 + (size_t)2 * H * sizeof(R1Term) + (size_t)8 * C * 8 +
                          (size_t)2 * H * 4 + 8 + (2 + 2 * R1X_ST) * 8;
    if (smem_x <= 220 * 1024) {
      long long tiles = (N + TR - 1) / TR;
      int cap = coda_sm_count();
      if (ctas_per_sm >= 1 && ctas_per_sm < 8) cap = cap - cap / 8;   // a concurrent stream keeps a few SMs
      int gridx = (int)min(tiles, (long long)cap);
#define LAUNCH_R1X(KC)                                                                                              \
  do {                                                                                                              \
    CODA_CUDA_OK(cudaFuncSetAttribute(k_pi_rank1_tma<KC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_x)); \
    k_pi_rank1_tma<KC><<<gridx, R1X_THREADS, smem_x, st>>>(preds, ens, N, C, TR, reinterpret_cast<const long long*>(sel), \
                                                          hdr, tlist, (float)lr, exp2f((float)fx_shift), U,        \
                                                          reinterpret_cast<unsigned long long*>(pisum_fx), flags); \
  } while (0)
      if (C <= 32) LAUNCH_R1X(1);
      else if (C <= 64) LAUNCH_R1X(2);
      else LAUNCH_R1X(4);
#undef LAUNCH_R1X
      CODA_LAUNCH_OK("k_pi_rank1_tma");
      return CODA_B200_OK;
    }
  }
  size_t smem = (size_t)8 * C * 8 + (size_t)2 * H * sizeof(R1Term);
  CODA_CHECK_ARG(smem <= 200 * 1024, "pi_rank1: C=%d too large", C);
  if constexpr (sizeof(T) == 4) if (!want_v1 && C <= 128) {
    long long want4 = (N + 8 * R1V_WI - 1) / (8 * R1V_WI);
    int cps = (ctas_per_sm < 1 || ctas_per_sm > 8) ? 8 : ctas_per_sm;
    int grid4 = (int)min(want4, (long long)coda_sm_count() * cps);
#define LAUNCH_R1V(KC)                                                                                            \
  do {                                                                                                            \
    CODA_CUDA_OK(cudaFuncSetAttribute(k_pi_rank1_v4<KC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    k_pi_rank1_v4<KC><<<grid4, 256, smem, st>>>(preds, ens, N, C, reinterpret_cast<const long long*>(sel), hdr,   \
                                               tlist, (float)lr, exp2f((float)fx_shift), U,                       \
                                               reinterpret_cast<unsigned long long*>(pisum_fx), flags);           \
  } while (0)
    if (C <= 32) LAUNCH_R1V(1);
    else if (C <= 64) LAUNCH_R1V(2);
    else LAUNCH_R1V(4);
#undef LAUNCH_R1V
    CODA_LAUNCH_OK("k_pi_rank1_v4");
    return CODA_B200_OK;
  }
  long long want = (N + R1_TN - 1) / R1_TN;
  if (ctas_per_sm < 1 || ctas_per_sm > 8) ctas_per_sm = 8;
  int grid = (int)min(want, (long long)coda_sm_count() * ctas_per_sm);
  // constant-bank slot of this caller (see c_terms_bank): the list is copied device-to-device on the launching stream
  const int slot_terms = (2 * H + 63) / 64 * 64;
  const bool use_const = const_slot >= 0 && (long long)(const_slot + 1) * slot_terms <= R1_CONST_TERMS && C <= 128;
  const int const_base = use_const ? const_slot * slot_terms : 0;
  if (use_const)
    CODA_CUDA_OK(cudaMemcpyToSymbolAsync(c_terms_bank, tlist, (size_t)2 * H * sizeof(R1Term),
                                         (size_t)const_base * sizeof(R1Term), cudaMemcpyDeviceToDevice, st));
#define LAUNCH_R1(KC)                                                                                          \
  do {                                                                                                         \
    if (use_const) {                                                                                           \
      CODA_CUDA_OK(cudaFuncSetAttribute(k_pi_rank1<T, KC, 16, 4, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
      k_pi_rank1<T, KC, 16, 4, true><<<grid, 256, smem, st>>>(preds, ens, N, C, reinterpret_cast<const long long*>(sel), hdr, \
                                            tlist, const_base, (float)lr, exp2f((float)fx_shift), U,           \
                                            reinterpret_cast<unsigned long long*>(pisum_fx), flags);           \
      break;                                                                                                   \
    }                                                                                                          \
    CODA_CUDA_OK(cudaFuncSetAttribute(k_pi_rank1<T, KC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    k_pi_rank1<T, KC><<<grid, 256, smem, st>>>(preds, ens, N, C, reinterpret_cast<const long long*>(sel), hdr,    \
                                            tlist, 0, (float)lr, exp2f((float)fx_shift), U,                    \
                                            reinterpret_cast<unsigned long long*>(pisum_fx), flags);           \
  } while (0)
  if (want_deep && C > 64 && C <= 128) {
    CODA_CUDA_OK(cudaFuncSetAttribute(k_pi_rank1<T, 4, 32, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_pi_rank1<T, 4, 32, 8><<<grid, 256, smem, st>>>(preds, ens, N, C, reinterpret_cast<const long long*>(sel), hdr, tlist, 0,
                                                  (float)lr, exp2f((float)fx_shift), U,
                                                  reinterpret_cast<unsigned long long*>(pisum_fx), flags);
    CODA_LAUNCH_OK("k_pi_rank1<deep>");
    return CODA_B200_OK;
  }
  if (C <= 32) LAUNCH_R1(1);
  else if (C <= 64) LAUNCH_R1(2);
  else if (C <= 128) LAUNCH_R1(4);
  else LAUNCH_R1(0);
#undef LAUNCH_R1
  CODA_LAUNCH_OK("k_pi_rank1");
  return CODA_B200_OK;
}

extern "C" int coda_b200_pi_rank1(const float* preds, const float* ens, int H, int64_t N, int C, const int64_t* sel,
                                  double lr, int fx_shift, const int32_t* terms /*[2 + 8H]*/, float* U,
                                  int64_t* pisum_fx, uint32_t* flags, int ctas_per_sm, int const_slot,
                                  coda_stream_t stream) {
  return pi_rank1(preds, ens, H, N, C, sel, lr, fx_shift, terms, U, pisum_fx, flags, ctas_per_sm, const_slot, stream);
}

extern "C" int coda_b200_pi_rank1_f16(const uint16_t* preds, const float* ens, int H, int64_t N, int C,
                                      const int64_t* sel, double lr, int fx_shift, const int32_t* terms, float* U,
                                      int64_t* pisum_fx, uint32_t* flags, int ctas_per_sm, int const_slot,
                                      coda_stream_t stream) {
  return pi_rank1(reinterpret_cast<const __half*>(preds), ens, H, N, C, sel, lr, fx_shift, terms, U, pisum_fx, flags,
                  ctas_per_sm, const_slot, stream);
}
