// K6 on the 5th-generation tensor cores: the MFCC-trajectory modulation spectrum as one GEMM.
//
// For a window x[0..win) of one coefficient trajectory (oracle: modulation_spectrum; north_star extension,
// SURVEY Appendix B) the kernel needs |rfft((x - mean) * hann, nfft)|.  Windowing and the DFT are one linear
// map, so with G[k][n] = hann[k] * {cos, -sin}(2 pi k n / nfft) the spectrum of 128 windows at once is
//
//     D[128 rows x nfft] = A[128 x K] . G[K x nfft],    A = mean-removed rows, K = win padded to 16,
//
// Re X[0 .. nfft/2] and Im X[1 .. nfft/2 - 1] (Im X[0] = Im X[nfft/2] = 0), i.e. exactly nfft output columns.
// Issued as tcgen05.mma kind::f16 with fp16 operand pairs (x s = hi + lo / 2048, G = Ghi + Glo / 2048, s a power
// of two per row; the low parts are carried at 2^11 so that they stay normal fp16 numbers): D0 = hi.Ghi and
// D1 = hi.Glo + lo.Ghi (result D0 + D1 / 2048) in SEPARATE fp32 accumulators in tensor memory -- the tensor core
// truncates when it adds into an accumulator, and 21 sequential adds into one accumulator biased the band
// energies by -1.4e-6 (measured); with the small terms apart the large one sees 7 adds.  To fit D0, D1 and A in
// 256 TMEM columns (two CTAs per SM) the bins go in two halves of 32: per half one N = 128 MMA per K slab
// (A_hi against [Ghi_half ; Glo_half] -> D0 | D1) plus one N = 64 MMA (A_lo against Ghi_half -> D1).
// A is written straight from registers into tensor memory (tcgen05.st, one TMEM lane per row), G is resident
// in shared memory in the canonical K-major layout.  Descriptor formats and the split's
// accuracy: tools/ubench/tcgen05_f16.cu, tools/ubench/tcgen05_tf32.cu (A from TMEM), tests/studies/tf32_dft_study.py.
//
// One CTA per (clip, chunk of windows) as in modspec_clip_kernel, rows in blocks of 128 ordered
// (coefficient, window) so that consecutive rows are consecutive output rows; the per-row-block shared buffer
// first stages the trajectories (coalesced loads), then the |X|^2 rows for band sums and coalesced stores.
#include <cuda_fp16.h>

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <type_traits>
#include <vector>

#include "mmf_internal.h"

namespace mmf {

namespace {

constexpr int kMtRows = 128;      // rows (trajectory windows) per block = the M of the MMA
constexpr int kMtThreads = 256;   // two threads per row: K halves in the operand preparation, bin halves in the epilogue
constexpr int kMtKMax = 128;  // win <= 128
constexpr long kMtSmemLimit = 110 * 1024;  // dynamic shared memory per CTA (two CTAs per SM)

__device__ __forceinline__ uint32_t mt_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ uint64_t mt_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
  uint64_t d = (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)((lbo >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo >> 4) & 0x3FFFu) << 32;
  d |= 1ull << 46;
  return d;
}

// A from tensor memory (lane = row, 32-bit column j = halves 2j, 2j+1), B from shared memory, fp16 -> fp32
__device__ __forceinline__ void mt_mma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, {%5, %5, %5, %5}, p;\n\t"
      "}\n" ::"r"(d_tmem),
      "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(acc), "r"(0u)
      : "memory");
}

__device__ __forceinline__ void mt_mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok = 0;
  while (!ok) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}\n"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
  }
}

__device__ __forceinline__ void mt_tmem_ld16(uint32_t taddr, float* v) {
  uint32_t* u = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]), "=r"(u[8]),
        "=r"(u[9]), "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15])
      : "r"(taddr)
      : "memory");
}

__device__ __forceinline__ void mt_tmem_st8(uint32_t taddr, const uint32_t* v) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr), "r"(v[0]),
               "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
               : "memory");
}

}  // namespace

struct ModTcArgs {
  const float* mfcc;
  int n_coef;
  long T;
  int win, hop;
  long n_win;
  int wc, n_chunks;
  long n_work;       // n_clips * n_chunks (VARLEN: the batch's items)
  int kp;            // win rounded up to 16
  const __half* g;   // [Ghi | Glo], each canonical K-major [NFFT rows x kp]
  float* mag;
  float* band;
  const int* band_lo;
  const int* band_hi;
  int n_bands;
  const ModItem* items;  // VARLEN: the batch's work items; T is then the row pitch, n_win the output window pitch
};

// half h, slot j (0..63): j < 32 -> Re X[32 h + j]; j >= 32 -> Im X[32 h + j - 32], except (h = 0, j = 32),
// whose Im X[0] = 0 slot carries Re X[nfft / 2].  VARLEN: a ragged batch, work item = p.items[item] (the default
// instantiation derives it from the item index and carries none of the ragged addressing).
template <int NFFT, int KS, bool VARLEN>
__global__ void __launch_bounds__(kMtThreads, 2) modspec_tc_kernel(const ModTcArgs p) {
  static_assert(NFFT == 128, "two halves of 32 bins");
  constexpr int nb = NFFT / 2 + 1;  // odd: conflict-free row pitch of the staging buffer
  constexpr int H = NFFT / 2;
  extern __shared__ __align__(1024) unsigned char sm_mt[];
  const int g_bytes = NFFT * p.kp * 2;
  __half* sGh = reinterpret_cast<__half*>(sm_mt);
  __half* sGl = reinterpret_cast<__half*>(sm_mt + g_bytes);
  float* s_buf = reinterpret_cast<float*>(sm_mt + 2 * g_bytes);          // [128][nb]: trajectories, then |X|^2 rows
  float** s_dst = reinterpret_cast<float**>(s_buf + kMtRows * nb);       // [128] output row pointers (128 * nb * 4 bytes: 8-byte aligned)
  float* s_iband = reinterpret_cast<float*>(s_dst + kMtRows);            // [wc * n_coef][n_bands]
  __shared__ float s_part[2][kMtRows];  // the two halves of a row's sum, then of its maximum
  __shared__ __align__(8) unsigned long long bar;
  __shared__ uint32_t tmem_base;
  __shared__ int s_blo[16], s_bhi[16];

  const int tid = threadIdx.x, warp = tid >> 5;
  // thread -> (row of the block, half): warps 0-3 and 4-7 own the same four TMEM lane quarters (warp & 3), so the two
  // threads of a row sit in warps w and w + 4 and can both reach the row's lane
  const int rr = tid & (kMtRows - 1), half = tid >> 7;

  for (int i = tid; i < 2 * g_bytes / 16; i += kMtThreads)
    reinterpret_cast<uint4*>(sm_mt)[i] = reinterpret_cast<const uint4*>(p.g)[i];
  if (tid < 16) {
    s_blo[tid] = tid < p.n_bands ? p.band_lo[tid] : 0;
    s_bhi[tid] = tid < p.n_bands ? p.band_hi[tid] : 0;
  }
  constexpr int kCols = NFFT + kMtKMax;  // D | A hi (kp/2 columns) | A lo (kp/2 columns)
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(mt_smem_u32(&tmem_base)), "r"(kCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (tid == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(mt_smem_u32(&bar)) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t d_tm = tmem_base, ah_tm = tmem_base + NFFT, al_tm = ah_tm + kMtKMax / 2;
  const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
  const uint32_t bar_a = mt_smem_u32(&bar);
  uint32_t parity = 0;
  const uint32_t sbo = (uint32_t)(p.kp / 8) * 128;
  // shared table: half 0 rows [Ghi_0 (64) ; Glo_0 (64)], then half 1 rows [Ghi_1 ; Glo_1]
  const uint64_t g_desc0 = mt_desc(mt_smem_u32(sGh), 128, sbo);
  const uint64_t g_desc1 = mt_desc(mt_smem_u32(sGl), 128, sbo);
  // fp16 x fp16 -> fp32, A and B K-major, M = 128
  const uint32_t idesc128 = (1u << 4) | ((uint32_t)(128 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
  const uint32_t idesc64 = (1u << 4) | ((uint32_t)(64 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
  constexpr int k_slabs = KS;
  const float inv_win = 1.0f / (float)p.win;

  // persistent: the 57 KB operand table is loaded once per CTA, then (clip, chunk) work items round-robin
  for (long item = blockIdx.x; item < p.n_work; item += gridDim.x) {
  long clip, w0, n_win_clip;  // n_win_clip: the clip's windows (p.n_win is the output pitch)
  int wca;
  if constexpr (VARLEN) {
    const ModItem it = p.items[item];
    clip = it.clip;
    w0 = it.w0;
    wca = it.wca;
    n_win_clip = it.n_win;
  } else {
    clip = item / p.n_chunks;
    const int chunk = (int)(item - clip * p.n_chunks);
    w0 = (long)chunk * p.wc;
    wca = (int)min((long)p.wc, p.n_win - w0);
    n_win_clip = p.n_win;
  }
  const int n_items = wca * p.n_coef;
  const int span = (wca - 1) * p.hop + p.win;
  for (int r0 = 0; r0 < n_items; r0 += kMtRows) {
    // ---- stage the trajectories this row block touches (coefficients c_lo .. c_hi), coalesced
    const int c_lo = r0 / wca, c_hi = min(r0 + kMtRows - 1, n_items - 1) / wca;
    // whole clip in one chunk and the touched trajectories fit with their own pitch T: one flat copy
    const int n_tr = c_hi - c_lo + 1;
    const bool flat_in = wca == n_win_clip && (long)n_tr * p.T <= (long)kMtRows * nb;
    const int pitch = flat_in ? (int)p.T : span;
    if (flat_in) {
      const float* src0 = p.mfcc + ((size_t)clip * p.n_coef + c_lo) * p.T;
      const int total = (n_tr - 1) * (int)p.T + span;
      constexpr int kBatch = 17;  // 2 x 17 x 256 >= 128 * nb
      for (int e0 = 0; e0 < total; e0 += kBatch * kMtThreads) {
        float a[kBatch];
#pragma unroll
        for (int u = 0; u < kBatch; ++u) {
          // clamped, not predicated: ptxas keeps a predicated load next to its store once it runs out of
          // predicate registers, which serialises the latencies
          const int e = min(e0 + u * kMtThreads + tid, total - 1);
          a[u] = __ldg(src0 + e);
        }
#pragma unroll
        for (int u = 0; u < kBatch; ++u) {
          const int e = e0 + u * kMtThreads + tid;
          if (e < total) s_buf[e] = a[u];
        }
      }
    } else {
      // eight independent loads per trajectory and thread in flight, four trajectories per step (the loads
      // of a step are all issued before its first store)
      const float* src0 = p.mfcc + ((size_t)clip * p.n_coef + c_lo) * p.T + w0 * p.hop;
      for (int c = 0; c < n_tr; c += 4) {
        const float* r0 = src0 + (size_t)c * p.T;
        const bool h1 = c + 1 < n_tr, h2 = c + 2 < n_tr, h3 = c + 3 < n_tr;
        const float* r1 = h1 ? r0 + p.T : r0;
        const float* r2 = h2 ? r0 + 2 * p.T : r0;
        const float* r3 = h3 ? r0 + 3 * p.T : r0;
        for (int i0 = 0; i0 < span; i0 += 8 * kMtThreads) {
          float a0[8], a1[8], a2[8], a3[8];
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const int i = i0 + u * kMtThreads + tid;
            const bool in = i < span;
            a0[u] = in ? __ldg(r0 + i) : 0.0f;
            a1[u] = (in && h1) ? __ldg(r1 + i) : 0.0f;
            a2[u] = (in && h2) ? __ldg(r2 + i) : 0.0f;
            a3[u] = (in && h3) ? __ldg(r3 + i) : 0.0f;
          }
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const int i = i0 + u * kMtThreads + tid;
            if (i < span) {
              s_buf[c * span + i] = a0[u];
              if (h1) s_buf[(c + 1) * span + i] = a1[u];
              if (h2) s_buf[(c + 2) * span + i] = a2[u];
              if (h3) s_buf[(c + 3) * span + i] = a3[u];
            }
          }
        }
      }
    }
    __syncthreads();
    // ---- two threads per row (K slabs [0, KH) and [KH, KS)): mean removal, power-of-two scale, fp16 split, A into
    // tensor memory.  The row's sum and maximum are combined through shared memory (same order in both threads).
    const int r = r0 + rr;
    const bool valid = r < n_items;
    const int coef = valid ? r / wca : c_lo;
    const int w = valid ? r - coef * wca : 0;
    float inv_s = 1.0f;
    {
      const float* x = s_buf + (coef - c_lo) * pitch + w * p.hop;
      // the two halves as two instantiations: slab ranges and the tail predicate are compile-time in each (a warp
      // lies in one half, so the branch is warp-uniform)
      auto prepare = [&](auto half_tag) {
        constexpr int HALF = decltype(half_tag)::value;
        constexpr int KH = (KS + 1) / 2;                 // slabs of half 0
        constexpr int K0 = HALF == 0 ? 0 : 16 * KH;      // first k of this half
        constexpr int NK = HALF == 0 ? 16 * KH : 16 * (KS - KH);
        float v[NK > 0 ? NK : 1];
        // mean removal relative to a pivot (the window's first sample): the differences are small next to a
        // trajectory's offset (c0 sits near -500), so the fp32 sum loses far less; four partial sums
        // rows past the last item read row (c_lo, 0): finite data, results never stored.  win > 16 (KS - 1):
        // only the last slab of the row needs the k < win predicate
        const float pivot = x[0];
        float sum4[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
        for (int kl = 0; kl < NK; ++kl) {
          const int k = K0 + kl;
          v[kl] = (k < 16 * KS - 16 || k < p.win) ? x[k] - pivot : 0.0f;
          sum4[kl & 3] += v[kl];
        }
        s_part[HALF][rr] = (sum4[0] + sum4[1]) + (sum4[2] + sum4[3]);
        __syncthreads();
        const float mean = (s_part[0][rr] + s_part[1][rr]) * inv_win;
        __syncthreads();  // both halves have read the sums: the buffer takes the maxima
        float m = 0.0f;
#pragma unroll
        for (int kl = 0; kl < NK; ++kl) {
          const int k = K0 + kl;
          v[kl] = (k < 16 * KS - 16 || k < p.win) ? v[kl] - mean : 0.0f;
          m = fmaxf(m, fabsf(v[kl]));
        }
        s_part[HALF][rr] = m;
        __syncthreads();
        m = fmaxf(s_part[0][rr], s_part[1][rr]);
        int e = (int)((__float_as_uint(m) >> 23) & 0xffu) - 127;
        if (m < 1e-30f) e = 5;
        e = max(-100, min(100, e));
        const float s = __uint_as_float((uint32_t)(5 - e + 127) << 23);  // m s in [32, 64)
        inv_s = __uint_as_float((uint32_t)(e - 5 + 127) << 23);
#pragma unroll
        for (int kc = 0; kc < NK / 16; ++kc) {
          uint32_t hi[8], lo[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float a = v[16 * kc + 2 * j] * s, b = v[16 * kc + 2 * j + 1] * s;
            const __half2 h2 = __floats2half2_rn(a, b);  // a in the low half = element 2j of the column
            const float2 f2 = __half22float2(h2);
            const __half2 l2 = __floats2half2_rn((a - f2.x) * 2048.0f, (b - f2.y) * 2048.0f);
            hi[j] = *reinterpret_cast<const uint32_t*>(&h2);
            lo[j] = *reinterpret_cast<const uint32_t*>(&l2);
          }
          mt_tmem_st8(ah_tm + lane_base + K0 / 2 + 8 * kc, hi);
          mt_tmem_st8(al_tm + lane_base + K0 / 2 + 8 * kc, lo);
        }
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
      };
      if (half == 0)
        prepare(std::integral_constant<int, 0>{});
      else
        prepare(std::integral_constant<int, 1>{});
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();  // A complete; the staged trajectories are dead from here on
    float* prow = s_buf + rr * nb;
    const float i2 = inv_s * inv_s;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      if (tid == 0) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint64_t gd = h == 0 ? g_desc0 : g_desc1;
#pragma unroll
        for (int s = 0; s < KS; ++s) mt_mma_ts(d_tm, ah_tm + 8 * s, gd + 16 * s, idesc128, s > 0 ? 1u : 0u);
#pragma unroll
        for (int s = 0; s < KS; ++s) mt_mma_ts(d_tm + 64, al_tm + 8 * s, gd + 16 * s, idesc64, 1u);
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar_a) : "memory");
      }
      mt_mbar_wait(bar_a, parity);
      parity ^= 1u;
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      // ---- |X|^2 of this thread's row, bins 32 h + 16 q .. + 15 with q = the thread's half, into the staging buffer
      // (pitch nb, odd)
      {
        const int q = half;
        float re0[16], re1[16], im0[16], im1[16];
        mt_tmem_ld16(d_tm + lane_base + 16 * q, re0);            // D0: hi . Ghi
        mt_tmem_ld16(d_tm + lane_base + 64 + 16 * q, re1);       // D1: hi . Glo + lo . Ghi
        mt_tmem_ld16(d_tm + lane_base + 32 + 16 * q, im0);
        mt_tmem_ld16(d_tm + lane_base + 96 + 16 * q, im1);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const float re = fmaf(re1[j], 1.0f / 2048.0f, re0[j]), im = fmaf(im1[j], 1.0f / 2048.0f, im0[j]);
          const int k = 32 * h + 16 * q + j;
          if (h == 0 && j == 0 && q == 0) {
            prow[0] = re * re * i2;
            prow[H] = im * im * i2;  // Re X[H] rides in the Im X[0] slot
          } else {
            prow[k] = (re * re + im * im) * i2;
          }
        }
      }
      if (h == 0) {
        // the next half overwrites D: every thread's loads must have completed
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
      }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();  // a row's |X|^2 values come from both of its threads
    {
      if (valid && p.n_bands > 0) {
        for (int b = half; b < p.n_bands; b += 2) {
          float e = 0.0f;
          for (int k = s_blo[b]; k < s_bhi[b]; ++k) e += prow[k];
          s_iband[((size_t)w * p.n_coef + coef) * p.n_bands + b] = e;
        }
      }
      if (half == 0)
        s_dst[rr] = (valid && p.mag != nullptr) ? p.mag + (((size_t)clip * p.n_coef + coef) * p.n_win + w0 + w) * nb : nullptr;
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    // ---- magnitudes out: rows are contiguous in memory wherever the coefficient does not change
    if (p.mag != nullptr && wca == p.n_win) {
      // the whole clip is one chunk: consecutive rows are consecutive output rows, the block is one flat
      // stream of min(128, n_items - r0) * nb floats
      float* dst = p.mag + (((size_t)clip * p.n_coef) * p.n_win + r0) * nb;
      const int n_out = min(kMtRows, n_items - r0) * nb;
#pragma unroll 13
      for (int e = tid; e < n_out; e += kMtThreads) {
        float m;
        asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(m) : "f"(s_buf[e]));
        dst[e] = m;
      }
    } else if (p.mag != nullptr) {
      // a warp writes its 16 rows one after the other, 65 consecutive floats per row; lane l (mod 16) holds row
      // l's destination and hands it round by shuffle (no dependent shared-memory load per row)
      const int lane = tid & 31;
      const unsigned long long mine = (unsigned long long)(uintptr_t)s_dst[warp * 16 + (lane & 15)];
#pragma unroll 4
      for (int q = 0; q < 16; ++q) {
        float* dst = reinterpret_cast<float*>((uintptr_t)__shfl_sync(0xffffffffu, mine, q));
        const float* src = s_buf + (warp * 16 + q) * nb;
        if (dst != nullptr) {
#pragma unroll
          for (int k0 = 0; k0 < nb; k0 += 32) {
            const int k = k0 + lane;
            if (k < nb) {
              float m;
              asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(m) : "f"(src[k]));
              dst[k] = m;
            }
          }
        }
      }
    }
    __syncthreads();
  }

  if (p.n_bands > 0) {
    // band energy of a window = sum over coefficients, fixed order (same as modspec_clip_kernel)
    for (int i = tid; i < wca * p.n_bands; i += kMtThreads) {
      const int w = i / p.n_bands, b = i - w * p.n_bands;
      float acc = 0.0f;
      for (int c = 0; c < p.n_coef; ++c) acc += s_iband[((size_t)w * p.n_coef + c) * p.n_bands + b];
      p.band[((size_t)clip * p.n_win + w0 + w) * p.n_bands + b] = acc;
    }
    __syncthreads();  // the band table is rewritten by the next work item
  }
  }  // work items
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0)
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kCols) : "memory");
}

// ---------------------------------------------------------------------------------------------------
// host
// ---------------------------------------------------------------------------------------------------
bool modspec_tc_supported(int win, int nfft) { return nfft == 128 && win >= 2 && win <= kMtKMax && win <= nfft; }

// Two half blocks of 128 rows x kp halves each, canonical K-major
// ((n / 8) * (kp / 8) * 64 + (k / 8) * 64 + (n % 8) * 8 + (k % 8)); in half h rows 0..63 = Ghi, rows 64..127 = Glo
// of slot j: j < 32 -> Re X[32 h + j], j >= 32 -> Im X[32 h + j - 32], (h = 0, j = 32) -> Re X[nfft / 2]
void modspec_tc_table(int win, int nfft, std::vector<uint16_t>& g, int* kp_out) {
  const int kp = (win + 15) / 16 * 16;
  const double kPi = 3.14159265358979323846;
  g.assign((size_t)2 * nfft * kp, 0);
  auto bits = [](__half h) {
    uint16_t u;
    std::memcpy(&u, &h, 2);
    return u;
  };
  auto idx = [&](int n, int k) { return (size_t)(n / 8) * (kp / 8) * 64 + (size_t)(k / 8) * 64 + (n % 8) * 8 + (k % 8); };
  for (int h = 0; h < 2; ++h)
    for (int j = 0; j < 64; ++j) {
      bool is_re = j < 32;
      int bin = 32 * h + (j & 31);
      if (h == 0 && j == 32) {
        is_re = true;
        bin = nfft / 2;
      }
      for (int k = 0; k < win; ++k) {
        const double hann = 0.5 - 0.5 * std::cos(2.0 * kPi * (double)k / (double)win);
        const long q = ((long)k * bin) % nfft;  // exact angle reduction
        const double ang = 2.0 * kPi * (double)q / (double)nfft;
        const double val = is_re ? hann * std::cos(ang) : -hann * std::sin(ang);
        const __half hi = __float2half_rn((float)val);
        const __half lo = __float2half_rn((float)((val - (double)__half2float(hi)) * 2048.0));
        g[idx(h * 128 + j, k)] = bits(hi);
        g[idx(h * 128 + 64 + j, k)] = bits(lo);
      }
    }
  *kp_out = kp;
}

// windows per CTA for one clip of T frames (0: the kernel does not take it): the whole clip if its band table fits,
// else chunks; a row block's trajectories (at most 128 / wc + 2 of them) must fit in the 128 x nb staging buffer
long modspec_tc_chunk(int win, int hop, int nfft, int n_coef, int n_bands, long T) {
  if (!modspec_tc_supported(win, nfft) || T < win || hop < 1) return 0;
  const int nb = nfft / 2 + 1;
  const int kp = (win + 15) / 16 * 16;
  const long n_win = 1 + (T - win) / hop;
  long wc = n_win;
  auto fits = [&](long w) {
    const long span = (w - 1) * hop + win;
    const long n_tr = std::min<long>(n_coef, (kMtRows - 1) / w + 2);
    // dynamic shared memory of a CTA: operand table + staging buffer + row pointers + band table, within the
    // 110 KB the kernel opts into (two CTAs per SM) less its static variables
    const long fixed = 2L * nfft * kp * 2 + (long)kMtRows * nb * 4 + (long)kMtRows * (long)sizeof(float*);
    return n_tr * span <= (long)kMtRows * nb && fixed + w * n_coef * std::max(n_bands, 1) * 4 <= kMtSmemLimit - 2048;
  };
  while (wc > 1 && !fits(wc)) wc = (wc + 1) / 2;
  if (!fits(wc)) return 0;
  const long n_chunks = (n_win + wc - 1) / wc;
  if (!fits(n_win - (n_chunks - 1) * wc)) return 0;  // the last chunk has fewer windows per coefficient
  return wc;
}

cudaError_t modspec_tc_launch(const float* mfcc, long n_clips, int n_coef, long T, int win, int hop, int nfft,
                              const void* g, int kp, long wc, float* mag, float* band, const int* lo, const int* hi,
                              int n_bands, int sm_count, cudaStream_t st, const ModVarlen* vl) {
  const int nb = nfft / 2 + 1;
  // T: frames per input row; n_win: windows per output row (a ragged batch: the row pitch and the most windows)
  const long n_win = vl ? vl->n_win : 1 + (T - win) / hop;
  const long n_chunks = (n_win + wc - 1) / wc;
  ModTcArgs a{};
  a.mfcc = mfcc;
  a.n_coef = n_coef;
  a.T = T;
  a.win = win;
  a.hop = hop;
  a.n_win = n_win;
  a.wc = (int)wc;
  a.n_chunks = (int)n_chunks;
  a.n_work = vl ? vl->n_items : n_clips * n_chunks;
  a.items = vl ? vl->items : nullptr;
  a.kp = kp;
  a.g = reinterpret_cast<const __half*>(g);
  a.mag = mag;
  a.band = band;
  a.band_lo = lo;
  a.band_hi = hi;
  a.n_bands = n_bands;
  const long wc_smem = vl ? vl->wc_max : wc;
  const size_t smem = (size_t)2 * nfft * kp * 2 + (size_t)kMtRows * nb * 4 + kMtRows * sizeof(float*) +
                      (size_t)wc_smem * n_coef * std::max(n_bands, 1) * 4;
  const unsigned grid = (unsigned)std::min<long>(a.n_work, 2L * sm_count);
#define MMF_MT_LAUNCH(KS, V)                          \
  {                                                   \
    auto kfn = modspec_tc_kernel<128, KS, V>;         \
    MMF_SMEM_ONCE(kfn, kMtSmemLimit);                 \
    kfn<<<grid, kMtThreads, smem, st>>>(a);           \
  }
#define MMF_MT_CASE(KS)                 \
  case KS: {                            \
    if (vl) MMF_MT_LAUNCH(KS, true)     \
    else MMF_MT_LAUNCH(KS, false)       \
    break;                              \
  }
  switch (kp / 16) {
    MMF_MT_CASE(1)
    MMF_MT_CASE(2)
    MMF_MT_CASE(3)
    MMF_MT_CASE(4)
    MMF_MT_CASE(5)
    MMF_MT_CASE(6)
    MMF_MT_CASE(7)
    MMF_MT_CASE(8)
    default: return cudaErrorInvalidValue;
  }
#undef MMF_MT_CASE
#undef MMF_MT_LAUNCH
  count_launch();
  return cudaGetLastError();
}

}  // namespace mmf
