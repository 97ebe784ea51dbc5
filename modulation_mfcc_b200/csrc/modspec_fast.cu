// K6 (fast path): modulation spectrum of the MFCC trajectories with the same
// register-resident mixed-radix FFT as the STFT kernel (SURVEY.md Appendix B).
//
// One "slot" of TPF = nfft/32 threads transforms one (clip, coefficient, window)
// trajectory window: 32 real samples per thread straight from global memory
// (the MFCC tensor is small and L2 resident), mean removal with a shuffle
// reduction over the slot, periodic Hann, zero padding to nfft, real FFT
// (16 x R2 x R3 passes, shared-memory exchange), |X| out, and the per-band
// energies reduced over the warp with shuffles.  A CTA owns one (clip, window)
// pair at a time: slot s takes coefficients s, s + SLOTS, ... in order, each warp
// accumulates its band sums in shared memory, and the warps' sums are added in
// warp order -- a fixed order, so the energies depend neither on scheduling nor
// on the batch a clip came in.
#include <cfloat>
#include <type_traits>

#include "mmf_internal.h"
#include "stft_core.cuh"

namespace mmf {

constexpr int kModThreads = 256;

template <int NFFT>
__global__ void __launch_bounds__(kModThreads)
    modspec_fast_kernel(const float* __restrict__ mfcc, int n_coef, long T, int win, int hop, long n_win, long n_pairs,
                        const float* __restrict__ hann, const float2* __restrict__ g_tw1,
                        const float2* __restrict__ g_tw2, float* __restrict__ mag, float* __restrict__ band,
                        const int* __restrict__ band_lo, const int* __restrict__ band_hi, int n_bands) {
  using C = FftCfg<NFFT>;
  static_assert(C::TPF <= 32, "one slot must fit in a warp");
  constexpr int SLOTS = kModThreads / C::TPF;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float2* s_xb = reinterpret_cast<float2*>(smem_raw);  // [SLOTS][XBUF]
  float2* s_tw1 = s_xb + SLOTS * C::XSTRIDE;              // [TW1]
  float2* s_tw2 = s_tw1 + C::TW1;                      // [TW2]
  __shared__ int s_blo[16], s_bhi[16];
  __shared__ float s_band[kModThreads / 32][16];  // per-warp band sums of the current pair
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int tau = tid % C::TPF, slot_in_block = tid / C::TPF;
  for (int i = tid; i < C::TW1; i += kModThreads) s_tw1[i] = g_tw1[i];
  for (int i = tid; i < C::TW2; i += kModThreads) s_tw2[i] = g_tw2[i];
  if (tid < 16) {
    s_blo[tid] = tid < n_bands ? band_lo[tid] : 0;
    s_bhi[tid] = tid < n_bands ? band_hi[tid] : 0;
  }
  float2 wreg[16];
#pragma unroll
  for (int n2 = 0; n2 < 16; ++n2) {
    const int c = tau + C::TPF * n2;
    wreg[n2] = make_float2(0.5f * hann[2 * c], 0.5f * hann[2 * c + 1]);  // zero beyond win
  }
  float2 wtau;
  sincospif(-2.0f * (float)tau / (float)NFFT, &wtau.y, &wtau.x);
  __syncthreads();

  float2* xb = s_xb + slot_in_block * C::XSTRIDE;
  const int nb = NFFT / 2 + 1;
  const float inv_win = 1.0f / (float)win;
  for (long pair = blockIdx.x; pair < n_pairs; pair += gridDim.x) {
  const long clip = pair / n_win, j = pair - clip * n_win;
  // every thread of the block runs the same number of iterations (the exchanges synchronise whole warps)
  for (int c0 = 0; c0 < n_coef; c0 += SLOTS) {
    const int coef = c0 + slot_in_block;
    const bool valid = coef < n_coef;
    const float* src = mfcc + ((size_t)clip * n_coef + coef) * T + j * hop;
    float2 v[16];
    float sum = 0.0f;
    // mean removal relative to a pivot (the window's first sample): next to a trajectory's offset (c0 sits
    // near -500) the differences are small, so the fp32 sum keeps its digits
    const float pivot = valid ? __ldg(src) : 0.0f;
#pragma unroll
    for (int n2 = 0; n2 < 16; ++n2) {
      const int i0 = 2 * (tau + C::TPF * n2);
      float x0 = 0.0f, x1 = 0.0f;
      if (valid) {
        if (i0 < win) x0 = __ldg(src + i0) - pivot;
        if (i0 + 1 < win) x1 = __ldg(src + i0 + 1) - pivot;
      }
      v[n2] = make_float2(x0, x1);
      sum += x0 + x1;
    }
#pragma unroll
    for (int o = C::TPF / 2; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    const float mean = sum * inv_win;
#pragma unroll
    for (int n2 = 0; n2 < 16; ++n2) v[n2] = make_float2((v[n2].x - mean) * wreg[n2].x, (v[n2].y - mean) * wreg[n2].y);

    ph_pass1<NFFT>(v, s_tw1, tau);
    __syncwarp();
    ph_x1_write<NFFT>(v, xb, tau);
    __syncwarp();
    ph_x1_read<NFFT>(v, xb, tau);
    ph_pass2<NFFT>(v, s_tw2, tau);
    if constexpr (C::R3 > 1) {
      __syncwarp();
      ph_x2_write<NFFT>(v, xb, tau);
      __syncwarp();
      ph_x2_read<NFFT>(v, xb, tau);
      ph_pass3<NFFT>(v);
    }
    __syncwarp();
    ph_z_write<NFFT>(v, xb, tau);
    __syncwarp();
    // power of this thread's bins -> registers, then (once every thread of the slot
    // has read its Z pairs) into shared memory in natural order, so that the
    // magnitude store and the band sums walk contiguous bins
    float pwr[17];
    {
      int q = 0;
      ph_split_smem_cb<NFFT>(xb, tau, wtau, [&](int, float p) { pwr[q++] = p; });
    }
    __syncwarp();
    float* pw = reinterpret_cast<float*>(xb);  // [nb] floats, aliases the exchange buffer
    {
      int q = 0;
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        const int k = tau + C::TPF * r;
        pw[k] = pwr[q++];
        pw[C::M - k] = pwr[q++];
      }
      if (tau == 0) pw[C::M / 2] = pwr[16];
    }
    __syncwarp();
    if (mag != nullptr && valid) {
      float* mdst = mag + (((size_t)clip * n_coef + coef) * n_win + j) * nb;
      for (int k = tau; k < nb; k += C::TPF) mdst[k] = sqrtf(pw[k]);
    }
    if (band != nullptr) {
      // invalid slots hold zeros
      for (int b = 0; b < n_bands; ++b) {
        float s = 0.0f;
        for (int k = s_blo[b] + tau; k < s_bhi[b]; k += C::TPF) s += pw[k];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) s_band[warp][b] = c0 == 0 ? s : s_band[warp][b] + s;
      }
    }
    __syncwarp();
  }
  if (band != nullptr) {
    __syncthreads();
    if (tid < n_bands) {
      float acc = 0.0f;
      for (int w = 0; w < kModThreads / 32; ++w) acc += s_band[w][tid];
      band[pair * n_bands + tid] = acc;
    }
    __syncthreads();  // s_band is rewritten by the next pair
  }
  }  // pairs
}

template <int NFFT>
static cudaError_t launch_t(const float* mfcc, long n_clips, int n_coef, long T, int win, int hop, const float* hann,
                            const float2* tw1, const float2* tw2, float* mag, float* band, const int* lo, const int* hi,
                            int n_bands, int sm_count, cudaStream_t st) {
  using C = FftCfg<NFFT>;
  const long n_win = 1 + (T - win) / hop;
  const long n_pairs = n_clips * n_win;
  const int slots = kModThreads / C::TPF;
  const long cap = (long)sm_count * 8;
  const long blocks = n_pairs < cap ? n_pairs : cap;
  const size_t smem = (size_t)(slots * C::XSTRIDE + C::TW1 + C::TW2 + 1) * sizeof(float2);
  MMF_SMEM_ONCE(modspec_fast_kernel<NFFT>, 200 * 1024);
  modspec_fast_kernel<NFFT><<<(unsigned)blocks, kModThreads, smem, st>>>(mfcc, n_coef, T, win, hop, n_win, n_pairs, hann,
                                                                      tw1, tw2, mag, band, lo, hi, n_bands);
  count_launch();
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// Clip-resident variant: one CTA per (clip, chunk of windows).  The chunk's span of
// every coefficient row is staged once in shared memory with coalesced loads (hop
// windows overlap, so nothing is re-read), the magnitudes of a pass go back to
// global memory as whole 4*(nfft/2+1)-byte rows, and the band energies are summed
// over coefficients in shared memory -- no scattered global accesses, no atomics.
// ---------------------------------------------------------------------------
// V = float2: one (window, coefficient) item per thread group; V = c2: two items per thread
// group on packed FP32 instructions (fft_regs.cuh), which halves the passes.  VARLEN: a ragged batch, the CTA's
// (clip, chunk) is items[blockIdx.x], T the input row pitch and n_win the output window pitch.
template <int NFFT, typename V, bool VARLEN>
__global__ void __launch_bounds__(kModThreads, 2)
    modspec_clip_kernel(const float* __restrict__ mfcc, int n_coef, long T, int win, int hop, long n_win, int wc,
                        int n_chunks, int pitch, const float* __restrict__ hann, const float2* __restrict__ g_tw1,
                        const float2* __restrict__ g_tw2, float* __restrict__ mag, float* __restrict__ band,
                        const int* __restrict__ band_lo, const int* __restrict__ band_hi, int n_bands,
                        const ModItem* __restrict__ items) {
  using C = FftCfg<NFFT>;
  using TR = CxTraits<V>;
  using Tw = typename TR::Tw;
  using Xe = typename TR::Xe;
  static_assert(C::TPF <= 32, "one slot must fit in a warp");
  constexpr int NI = TR::kFrames;  // items per thread group
  constexpr int SLOTS = kModThreads / C::TPF;
  constexpr int nb = NFFT / 2 + 1;
  constexpr int PWP = (nb + 1) & ~1;  // floats per item in a slot's power area
  static_assert(NI * PWP * 4 <= C::XBUF * 8, "power rows must fit in the exchange buffer of the slot");
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Xe* s_xb = reinterpret_cast<Xe*>(smem_raw);                      // [SLOTS][XBUF]
  Tw* s_tw1 = reinterpret_cast<Tw*>(s_xb + SLOTS * C::XSTRIDE);       // [TW1]
  Tw* s_tw2 = s_tw1 + C::TW1;                                      // [TW2 + 1]
  float2* s_win = reinterpret_cast<float2*>(s_tw2 + C::TW2 + 1);   // [M] half-scaled Hann pairs (zero beyond win)
  float* s_rows = reinterpret_cast<float*>(s_win + C::M);          // [n_coef][pitch]
  float* s_iband = s_rows + (size_t)n_coef * pitch;                // [wc * n_coef][n_bands]
  float** s_dst = reinterpret_cast<float**>(s_iband + (((size_t)wc * n_coef * n_bands + 1) & ~(size_t)1));  // [SLOTS*NI]
  __shared__ int s_blo[16], s_bhi[16];
  const int tid = threadIdx.x;
  const int tau = tid % C::TPF, slot = tid / C::TPF;
  long clip, w0;
  int wca;  // windows of this chunk
  if constexpr (VARLEN) {
    const ModItem it = items[blockIdx.x];
    clip = it.clip;
    w0 = it.w0;
    wca = it.wca;
  } else {
    clip = blockIdx.x / n_chunks;
    const int chunk = (int)(blockIdx.x - clip * n_chunks);
    w0 = (long)chunk * wc;
    wca = (int)min((long)wc, n_win - w0);
  }
  const int span = (wca - 1) * hop + win;

  for (int i = tid; i < C::TW1; i += kModThreads) s_tw1[i] = make_tw<V>(g_tw1[i]);
  for (int i = tid; i < C::TW2; i += kModThreads) s_tw2[i] = make_tw<V>(g_tw2[i]);
  for (int i = tid; i < C::M; i += kModThreads) s_win[i] = make_float2(0.5f * hann[2 * i], 0.5f * hann[2 * i + 1]);
  if (tid < 16) {
    s_blo[tid] = tid < n_bands ? band_lo[tid] : 0;
    s_bhi[tid] = tid < n_bands ? band_hi[tid] : 0;
  }
  {
    // stage the chunk's span of every coefficient row, two rows and four column blocks per step
    // (eight independent loads in flight per thread, no integer division)
    const float* src0 = mfcc + (size_t)clip * n_coef * T + w0 * hop;
    for (int c = 0; c < n_coef; c += 2) {
      const float* r0 = src0 + (size_t)c * T;
      const bool has1 = c + 1 < n_coef;
      const float* r1 = has1 ? r0 + T : r0;
      for (int i = tid; i < span; i += 4 * kModThreads) {
        float a[4], b[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int ii = i + u * kModThreads;
          a[u] = ii < span ? __ldg(r0 + ii) : 0.0f;
          b[u] = ii < span ? __ldg(r1 + ii) : 0.0f;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int ii = i + u * kModThreads;
          if (ii < span) {
            s_rows[c * pitch + ii] = a[u];
            if (has1) s_rows[(c + 1) * pitch + ii] = b[u];
          }
        }
      }
    }
  }
  Tw wtau;
  {
    float2 w;
    sincospif(-2.0f * (float)tau / (float)NFFT, &w.y, &w.x);
    wtau = make_tw<V>(w);
  }
  __syncthreads();

  Xe* xb = s_xb + slot * C::XSTRIDE;
  float* pw = reinterpret_cast<float*>(xb);  // [NI][PWP] power of this slot's items, aliases the exchange buffer
  const float inv_win = 1.0f / (float)win;
  const int n_items = wca * n_coef;  // item = window * n_coef + coefficient
  for (int base = 0; base < n_items; base += SLOTS * NI) {
    int item[NI];
    bool valid[NI];
    float xs[NI][32];
    float mean[NI];
#pragma unroll
    for (int q = 0; q < NI; ++q) {
      item[q] = base + slot * NI + q;
      valid[q] = item[q] < n_items;
      const int w = valid[q] ? item[q] / n_coef : 0;
      const int coef = valid[q] ? item[q] - w * n_coef : 0;
      const float* src = s_rows + coef * pitch + w * hop;
      float sum = 0.0f;
      const float pivot = valid[q] ? src[0] : 0.0f;  // see modspec_fast_kernel
#pragma unroll
      for (int n2 = 0; n2 < 16; ++n2) {
        const int i0 = 2 * (tau + C::TPF * n2);
        const float x0 = (valid[q] && i0 < win) ? src[i0] - pivot : 0.0f;
        const float x1 = (valid[q] && i0 + 1 < win) ? src[i0 + 1] - pivot : 0.0f;
        xs[q][2 * n2] = x0;
        xs[q][2 * n2 + 1] = x1;
        sum += x0 + x1;
      }
#pragma unroll
      for (int o = C::TPF / 2; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
      mean[q] = sum * inv_win;
      if (tau == 0)
        s_dst[slot * NI + q] =
            (mag != nullptr && valid[q]) ? mag + (((size_t)clip * n_coef + coef) * n_win + w0 + w) * nb : nullptr;
    }
    V v[16];
#pragma unroll
    for (int n2 = 0; n2 < 16; ++n2) {
      const float2 wv = s_win[tau + C::TPF * n2];
      if constexpr (NI == 1) {
        v[n2] = make_float2((xs[0][2 * n2] - mean[0]) * wv.x, (xs[0][2 * n2 + 1] - mean[0]) * wv.y);
      } else {
        v[n2] = CxTraits<c2>::make(pmake((xs[0][2 * n2] - mean[0]) * wv.x, (xs[1][2 * n2] - mean[1]) * wv.x),
                                   pmake((xs[0][2 * n2 + 1] - mean[0]) * wv.y, (xs[1][2 * n2 + 1] - mean[1]) * wv.y));
      }
    }

    ph_pass1<NFFT>(v, s_tw1, tau);
    if constexpr (TR::kXParts == 1) {
      __syncwarp();
      ph_x1_write<NFFT, 0>(v, xb, tau);
      __syncwarp();
      ph_x1_read<NFFT, 0>(v, xb, tau);
    } else {
      __syncwarp();
      ph_x1_write<NFFT, 1>(v, xb, tau);
      __syncwarp();
      ph_x1_read<NFFT, 1>(v, xb, tau);
      __syncwarp();
      ph_x1_write<NFFT, 2>(v, xb, tau);
      __syncwarp();
      ph_x1_read<NFFT, 2>(v, xb, tau);
    }
    ph_pass2<NFFT>(v, s_tw2, tau);
    if constexpr (C::R3 > 1) {
      if constexpr (TR::kXParts == 1) {
        __syncwarp();
        ph_x2_write<NFFT, 0>(v, xb, tau);
        __syncwarp();
        ph_x2_read<NFFT, 0>(v, xb, tau);
      } else {
        __syncwarp();
        ph_x2_write<NFFT, 1>(v, xb, tau);
        __syncwarp();
        ph_x2_read<NFFT, 1>(v, xb, tau);
        __syncwarp();
        ph_x2_write<NFFT, 2>(v, xb, tau);
        __syncwarp();
        ph_x2_read<NFFT, 2>(v, xb, tau);
      }
      ph_pass3<NFFT>(v);
    }
    V za[9], zb[8];
    if constexpr (TR::kXParts == 1) {
      __syncwarp();
      ph_z_write<NFFT, 0>(v, xb, tau);
      __syncwarp();
      ph_z_gather<NFFT, 0>(za, zb, xb, tau);
    } else {
      __syncwarp();
      ph_z_write<NFFT, 1>(v, xb, tau);
      __syncwarp();
      ph_z_gather<NFFT, 1>(za, zb, xb, tau);
      __syncwarp();
      ph_z_write<NFFT, 2>(v, xb, tau);
      __syncwarp();
      ph_z_gather<NFFT, 2>(za, zb, xb, tau);
    }
    __syncwarp();  // every thread of the slot has its Z pairs: the buffer becomes the power area
    // power rows in natural bin order: pw[q * PWP + k]
    {
      V pr[9];
#pragma unroll
      for (int r = 0; r < 8; ++r) pr[r] = split_pair(za[r], zb[r], w32(r), wtau);
      pr[8] = split_pair(za[8], za[8], w32(8), wtau);
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        const int k = tau + C::TPF * r;
        if constexpr (NI == 1) {
          pw[k] = pr[r].x;
          pw[C::M - k] = pr[r].y;
        } else {
          pw[k] = plo(pr[r].x);
          pw[PWP + k] = phi(pr[r].x);
          pw[C::M - k] = plo(pr[r].y);
          pw[PWP + C::M - k] = phi(pr[r].y);
        }
      }
      if (tau == 0) {
        if constexpr (NI == 1) {
          pw[C::M / 2] = pr[8].x;
        } else {
          pw[C::M / 2] = plo(pr[8].x);
          pw[PWP + C::M / 2] = phi(pr[8].x);
        }
      }
    }
    __syncwarp();
    if (band != nullptr) {  // (every lane takes part in the shuffles; invalid items just do not store)
#pragma unroll
      for (int q = 0; q < NI; ++q)
        for (int b = 0; b < n_bands; ++b) {
          float e = 0.0f;
          for (int k = s_blo[b] + tau; k < s_bhi[b]; k += C::TPF) e += pw[q * PWP + k];
#pragma unroll
          for (int o = C::TPF / 2; o > 0; o >>= 1) e += __shfl_xor_sync(0xffffffffu, e, o);
          if (tau == 0 && valid[q]) s_iband[(size_t)item[q] * n_bands + b] = e;
        }
    }
    __syncthreads();
    // whole magnitude rows of this pass: one warp per row, consecutive lanes -> consecutive bins
    if (mag != nullptr) {
      const int n_here = min(SLOTS * NI, n_items - base);
      const int lane = tid & 31;
      for (int it = tid >> 5; it < n_here; it += kModThreads / 32) {
        float* d = s_dst[it];
        const float* src = reinterpret_cast<const float*>(s_xb + (it / NI) * C::XSTRIDE) + (it % NI) * PWP;
        if (d != nullptr)
          for (int k = lane; k < nb; k += 32) d[k] = sqrtf(src[k]);
      }
    }
    __syncthreads();
  }
  if (band != nullptr) {
    for (int e = tid; e < wca * n_bands; e += kModThreads) {
      const int w = e / n_bands, b = e - w * n_bands;
      float acc = 0.0f;
      for (int c = 0; c < n_coef; ++c) acc += s_iband[((size_t)w * n_coef + c) * n_bands + b];
      band[((size_t)clip * n_win + w0 + w) * n_bands + b] = acc;
    }
  }
}

// the clip kernel's budget: its rows + per-item band sums within ~110 KB, so that two CTAs share an SM
template <int NFFT>
struct ClipSmem {
  using C = FftCfg<NFFT>;
  static constexpr int SLOTS = kModThreads / C::TPF;
  static constexpr int nb = NFFT / 2 + 1;
  // two items per thread group (packed FP32) when both power rows fit in the slot's exchange buffer
  static constexpr bool kPacked = 2 * ((nb + 1) & ~1) * 4 <= C::XBUF * 8;
  using V = typename std::conditional<kPacked, c2, float2>::type;
  static constexpr int NI = kPacked ? 2 : 1;
  static constexpr size_t kBudget = 110 * 1024;
  static size_t need(int n_coef, int win, int hop, int nbands, long w) {
    const size_t fixed = (size_t)SLOTS * C::XSTRIDE * 8 + (size_t)(C::TW1 + C::TW2 + 1) * sizeof(typename CxTraits<V>::Tw) +
                         (size_t)C::M * 8 + (size_t)SLOTS * NI * sizeof(float*) + 64;
    const long span = (w - 1) * hop + win;
    const long pitch = (span + 1) & ~1L;
    return fixed + (size_t)n_coef * pitch * 4 + ((((size_t)w * n_coef * nbands) + 1) & ~(size_t)1) * 4;
  }
};

// windows per CTA for one clip of T frames: as many as fit the budget (0: not even one fits, the fast kernel takes it)
template <int NFFT>
static long clip_chunk_t(int n_coef, int win, int hop, int nbands, long T) {
  using S = ClipSmem<NFFT>;
  const long n_win = 1 + (T - win) / hop;
  long wc = n_win;
  if (S::need(n_coef, win, hop, nbands, 1) > S::kBudget) return 0;
  while (wc > 1 && S::need(n_coef, win, hop, nbands, wc) > S::kBudget) wc = (wc + 1) / 2;
  while (wc < n_win && S::need(n_coef, win, hop, nbands, wc + 1) <= S::kBudget) ++wc;
  return wc;
}

template <int NFFT>
static cudaError_t launch_clip_t(const float* mfcc, long n_clips, int n_coef, long T, int win, int hop, long wc,
                                 const float* hann, const float2* tw1, const float2* tw2, float* mag, float* band,
                                 const int* lo, const int* hi, int n_bands, cudaStream_t st, const ModVarlen* vl) {
  using S = ClipSmem<NFFT>;
  const long n_win = vl ? vl->n_win : 1 + (T - win) / hop;
  const int nbands = band != nullptr ? n_bands : 0;
  const long wcs = vl ? vl->wc_max : wc;  // the largest chunk lays out shared memory
  const long n_chunks = (n_win + wc - 1) / wc;
  const long span = (wcs - 1) * hop + win;
  const int pitch = (int)((span + 1) & ~1L);
  const size_t smem = S::need(n_coef, win, hop, nbands, wcs);
  const unsigned grid = (unsigned)(vl ? vl->n_items : n_clips * n_chunks);
#define MMF_CLIP_LAUNCH(VL)                                                                                          \
  {                                                                                                                  \
    auto kfn = modspec_clip_kernel<NFFT, typename S::V, VL>;                                                         \
    MMF_SMEM_ONCE(kfn, 200 * 1024);                                                                                  \
    kfn<<<grid, kModThreads, smem, st>>>(mfcc, n_coef, T, win, hop, n_win, (int)wcs, (int)n_chunks, pitch, hann, tw1, \
                                         tw2, mag, band, lo, hi, n_bands, vl ? vl->items : nullptr);                 \
  }
  if (vl)
    MMF_CLIP_LAUNCH(true)
  else
    MMF_CLIP_LAUNCH(false)
#undef MMF_CLIP_LAUNCH
  count_launch();
  return cudaGetLastError();
}

bool modspec_fast_supported(int nfft) { return nfft >= 32 && nfft <= 1024; }

long modspec_clip_chunk(int win, int hop, int nfft, int n_coef, int n_bands, long T) {
  if (T < win || hop < 1) return 0;
  switch (nfft) {
    case 32: return clip_chunk_t<32>(n_coef, win, hop, n_bands, T);
    case 64: return clip_chunk_t<64>(n_coef, win, hop, n_bands, T);
    case 128: return clip_chunk_t<128>(n_coef, win, hop, n_bands, T);
    case 256: return clip_chunk_t<256>(n_coef, win, hop, n_bands, T);
    case 512: return clip_chunk_t<512>(n_coef, win, hop, n_bands, T);
    case 1024: return clip_chunk_t<1024>(n_coef, win, hop, n_bands, T);
    default: return 0;
  }
}

cudaError_t modspec_clip_launch(const float* mfcc, long n_clips, int n_coef, long T, int win, int hop, int nfft,
                                long wc, const float* hann, const float2* tw1, const float2* tw2, float* mag,
                                float* band, const int* lo, const int* hi, int n_bands, cudaStream_t st,
                                const ModVarlen* vl) {
#define MMF_MOD_CASE(N)                                                                                              \
  case N:                                                                                                            \
    return launch_clip_t<N>(mfcc, n_clips, n_coef, T, win, hop, wc, hann, tw1, tw2, mag, band, lo, hi, n_bands, st, vl);
  switch (nfft) {
    MMF_MOD_CASE(32)
    MMF_MOD_CASE(64)
    MMF_MOD_CASE(128)
    MMF_MOD_CASE(256)
    MMF_MOD_CASE(512)
    MMF_MOD_CASE(1024)
    default: return cudaErrorInvalidValue;
  }
#undef MMF_MOD_CASE
}

cudaError_t modspec_fast_launch(const float* mfcc, long n_clips, int n_coef, long T, int win, int hop, int nfft,
                                const float* hann, const float2* tw1, const float2* tw2, float* mag, float* band,
                                const int* lo, const int* hi, int n_bands, int sm_count, cudaStream_t st) {
  if (T < win) return cudaSuccess;
#define MMF_MOD_CASE(N) \
  case N: return launch_t<N>(mfcc, n_clips, n_coef, T, win, hop, hann, tw1, tw2, mag, band, lo, hi, n_bands, sm_count, st);
  switch (nfft) {
    MMF_MOD_CASE(32)
    MMF_MOD_CASE(64)
    MMF_MOD_CASE(128)
    MMF_MOD_CASE(256)
    MMF_MOD_CASE(512)
    MMF_MOD_CASE(1024)
    default: return cudaErrorInvalidValue;
  }
#undef MMF_MOD_CASE
}

void modspec_geometry(int nfft, StftGeometry* g) {
  g->m = nfft / 2;
  g->tpf = g->m / 16;
  const int r2 = g->tpf < 16 ? g->tpf : 16;
  g->r3 = g->tpf / r2;
  g->tw1 = 16 * g->tpf;
  g->tw2 = 16 * g->r3;
  g->fpi = 0;
}

}  // namespace mmf
