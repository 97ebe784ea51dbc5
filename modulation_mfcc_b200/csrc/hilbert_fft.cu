// Hilbert amplitude envelope |scipy.signal.hilbert(x)| in O(n log n) for any length n
// (script/calc.py:284-286, method 'Hilb': FFT of length n, negative frequencies zeroed, inverse FFT).
//
// scipy transforms at the signal's own length (160 000 for a 10 s clip, 57.6 M for an hour): not a power of
// two, often with large prime factors.  Bluestein's identity turns a length-n DFT into a circular convolution
// of length M = 2^m >= 2n - 1 with the chirp c[j] = exp(-i pi j^2 / n):
//     X[k] = c[k] * sum_j (x[j] c[j]) conj(c[k - j]).
// The convolutions run through a radix-2 Stockham FFT of length M (natural order in and out, twiddles from a
// table); chirp phases are reduced exactly (j^2 mod 2n in integer arithmetic).  Everything is float64 -- the
// result is then exact to ~1e-12 (scipy itself computes float32 input in single precision).
// Envelope = | IDFT_n( H . DFT_n(x) ) | with H = 1 (k = 0, and n/2 for even n), 2 (0 < k < n/2), 0 otherwise;
// the inverse transform reuses the forward machinery on conjugated data.
//
// Per clip that is five transforms: the chirp filter's (once per distinct n of a batch), then four on the clip:
//   1. a = x c (zero padded)                  -> FFT -> conj(. bf)
//   2.                                           FFT -> mask: conj(H c conj(.)/M) c for j < n, 0 past n
//   3.                                           FFT -> conj(. bf)
//   4.                                           FFT -> |c conj(.)| / (M n) for j < n
// Radix-2 Stockham pass p (Ns = 2^p) pairs elements j and j + M/2 (twiddle w[k M/2 / Ns], k = j mod Ns) and
// writes 2(j - k) + k and that + Ns.  Passes p0 .. p0 + L - 1 only mix elements that share every index bit but
// the top L of their input index; they leave them at [middle bits | L new bits | low p0 bits].  So a transform
// runs as 2 (m <= 22) or 3 pass groups of at most 11 bits, each one launch over every row of a batch: a CTA loads
// C = 4096 / 2^L such sub-transforms (consecutive in their low bits, so the strided loads coalesce) into shared
// memory, runs the L passes there and stores them.  The pointwise steps ride on the first and last groups.
//
// Every output is bit-identical to the former one-launch-per-pass kernels: each element sees the same
// operations in the same order.  The arithmetic is written with explicit __dmul_rn / __fma_rn / __dadd_rn so that
// fusion cannot change how the compiler contracts it; the forms mirror the SASS sm_100a made of those kernels
// (cmul_d as two DMUL then two DFMA, which products are rounded noted at each use).
#include <cmath>

#include "mmf_internal.h"

namespace mmf {

namespace {

constexpr int kLogE = 12;          // elements per CTA of a pass group: 2^12 double2 = 64 KB of shared memory
constexpr int kE = 1 << kLogE;
constexpr int kThreads = 512;      // four butterflies per thread and pass
constexpr float kq = 1.0f / 32768.0f;  // as pcm16_to_f32_kernel scales int16

// a * b with a.x b.y and a.y b.y rounded, a.x b.x and a.y b.x fused (the butterfly and conj(. bf) products)
__device__ __forceinline__ double2 cmul_rb(double2 a, double2 b) {
  return make_double2(__fma_rn(a.x, b.x, -__dmul_rn(a.y, b.y)), __fma_rn(a.y, b.x, __dmul_rn(a.x, b.y)));
}
// a * b with a.y b.x and a.y b.y rounded (the products with the chirp c = a in the mask and the envelope)
__device__ __forceinline__ double2 cmul_ra(double2 a, double2 b) {
  return make_double2(__fma_rn(b.x, a.x, -__dmul_rn(b.y, a.y)), __fma_rn(b.y, a.x, __dmul_rn(b.x, a.y)));
}

// c[j] = exp(-i pi j^2 / n), j < n, with j^2 reduced mod 2n exactly; one ragged launch over the distinct n
__global__ void hilbert_chirp_kernel(const HilRow* __restrict__ rows, const unsigned* __restrict__ first, long n_rows,
                                     double2* __restrict__ s) {
  long r = 0, hi = n_rows - 1;
  while (r < hi) {
    const long mid = (r + hi + 1) >> 1;
    if (first[mid] <= blockIdx.x) r = mid;
    else hi = mid - 1;
  }
  const HilRow& row = rows[r];
  const long j = (long)(blockIdx.x - first[r]) * blockDim.x + threadIdx.x, n = row.n;
  if (j >= n) return;
  const unsigned long long q = ((unsigned long long)j * (unsigned long long)j) % (unsigned long long)(2 * n);
  double sn, co;
  sincospi(-(double)q / (double)n, &sn, &co);
  s[row.c + j] = make_double2(co, sn);
}

// W[k] = exp(-2 pi i k / M), k < M/2, for the batch's largest M.  A row of length M' = M / 2^d reads entry k 2^d:
// sincospi(-(k 2^d) / (M/2)) receives the same double as sincospi(-k / (M'/2)) (both quotients are the correctly
// rounded value of one rational), so the entries are the ones a table built for M' would hold.
__global__ void hilbert_twiddle_kernel(long half, double2* __restrict__ w) {
  const long k = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= half) return;
  double sn, co;
  sincospi(-(double)k / (double)half, &sn, &co);
  w[k] = make_double2(co, sn);
}

// One pass group g of transform T (0: the chirp filter's, 1-4: the clip's) over the rows of a batch; a CTA is C
// sub-transforms of one row.  Shared layout: element t of sub-transform c at (t << logC) | (c ^ (t & (C - 1))).
__global__ void __launch_bounds__(kThreads, 2) hilbert_group_kernel(HilPass p) {
  extern __shared__ double2 sm[];
  long r = 0, hi = p.n_rows - 1;
  while (r < hi) {
    const long mid = (r + hi + 1) >> 1;
    if (p.first[mid] <= blockIdx.x) r = mid;
    else hi = mid - 1;
  }
  const HilRow row = p.rows[r];
  const int g = p.g, m = row.m, G = row.G;
  const int Lg = g == 0 ? row.L[0] : (g == 1 ? row.L[1] : row.L[2]), logC = kLogE - Lg, C = 1 << logC;
  const int p0 = g == 0 ? 0 : (g == 1 ? row.L[0] : row.L[0] + row.L[1]);
  const long M = 1L << m, n = row.n;
  const long r0 = (long)(blockIdx.x - p.first[r]) << logC;  // first sub-transform: its low m - Lg index bits
  auto sidx = [&](int t, int c) { return (t << logC) | (c ^ (t & (C - 1))); };
  // group step of the row: step s writes buf0 (s even) or buf1 and reads what step s - 1 wrote; the chirp filter's
  // last group writes buf0 = bf
  const int step = p.T == 0 ? g + ((G - 1) & 1) : (p.T - 1) * G + g;
  double2* __restrict__ dst = p.s + ((step & 1) ? row.buf1 : row.buf0);
  const double2* __restrict__ src = p.s + ((step & 1) ? row.buf0 : row.buf1);
  const double2* __restrict__ c = p.s + row.c;
  // ---- load: element t of sub-transform c is input index (t << (m - Lg)) + r0 + c
  for (int i = threadIdx.x; i < kE; i += kThreads) {
    const int cc = i & (C - 1), t = i >> logC;
    const long j = ((long)t << (m - Lg)) + r0 + cc;
    double2 v;
    if (g == 0 && p.T == 0) {  // b[j] = conj(c[|j|]) wrapped to length M
      v = make_double2(0.0, 0.0);
      if (j < n) v = make_double2(c[j].x, -c[j].y);
      else if (M - j < n) v = make_double2(c[M - j].x, -c[M - j].y);
    } else if (g == 0 && p.T == 1) {  // a[j] = x[j] c[j], zero padded
      v = make_double2(0.0, 0.0);
      if (j < n) {
        const double xv = p.pcm16 ? (double)((float)((const int16_t*)p.x)[row.src + j] * kq)
                                  : (double)((const float*)p.x)[row.src + j];
        const double2 cj = c[j];
        v = make_double2(__dmul_rn(xv, cj.x), __dmul_rn(xv, cj.y));
      }
    } else {
      v = src[j];
    }
    sm[sidx(t, cc)] = v;
  }
  __syncthreads();
  // ---- the group's passes: local pass s is global pass p0 + s, twiddle k = (k_loc << p0) | lo
  const long lo_mask = (1L << p0) - 1;
  const int hl = 1 << (Lg - 1);
  for (int s = 0; s < Lg; ++s) {
    const int Ns = 1 << s, sh = p.mw - 1 - p0 - s;
    double2 oa[kE / 2 / kThreads], ob[kE / 2 / kThreads];
    int ia[kE / 2 / kThreads], ib[kE / 2 / kThreads];
#pragma unroll
    for (int q = 0; q < kE / 2 / kThreads; ++q) {
      const int b = threadIdx.x + q * kThreads, cc = b & (C - 1), jl = b >> logC, k = jl & (Ns - 1);
      const double2 a = sm[sidx(jl, cc)], u = sm[sidx(jl + hl, cc)];
      const long tk = (((long)k << p0) | ((r0 + cc) & lo_mask)) << sh;
      const double2 t = cmul_rb(u, __ldg(p.w + tk));
      oa[q] = make_double2(__dadd_rn(a.x, t.x), __dadd_rn(a.y, t.y));
      ob[q] = make_double2(__dsub_rn(a.x, t.x), __dsub_rn(a.y, t.y));
      const int j0 = ((jl - k) << 1) + k;
      ia[q] = sidx(j0, cc);
      ib[q] = sidx(j0 + Ns, cc);
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < kE / 2 / kThreads; ++q) {
      sm[ia[q]] = oa[q];
      sm[ib[q]] = ob[q];
    }
    __syncthreads();
  }
  // ---- store: element u of sub-transform c is output index [mid | u | lo]; the last group applies the pointwise step
  const bool last = g == G - 1;
  const double2* __restrict__ bf = p.s + row.bf;
  const double inv_m = 1.0 / (double)M;  // a power of two: exact
  for (int i = threadIdx.x; i < kE; i += kThreads) {
    int cc, u;
    long y;
    if (p0 == 0) {  // contiguous: y = (r0 + c) 2^Lg + u
      cc = i >> Lg;
      u = i & ((1 << Lg) - 1);
      y = (r0 << Lg) + i;
    } else {  // contiguous in c
      cc = i & (C - 1);
      u = i >> logC;
      const long rr = r0 + cc;
      y = ((rr >> p0) << (p0 + Lg)) | ((long)u << p0) | (rr & lo_mask);
    }
    const double2 v = sm[sidx(u, cc)];
    if (!last || p.T == 0) {
      dst[y] = v;
    } else if (p.T == 1 || p.T == 3) {  // conj(v bf)
      const double2 q = cmul_rb(v, bf[y]);
      dst[y] = make_double2(q.x, -q.y);
    } else if (p.T == 2) {  // conv = conj(v) / M; X = c conv; next = conj(H X) c for y < n, zero past n
      double2 o = make_double2(0.0, 0.0);
      if (y < n) {
        const double2 cy = c[y];
        const double2 conv = make_double2(__dmul_rn(v.x, inv_m), __dmul_rn(v.y, -inv_m));
        const double2 X = cmul_ra(cy, conv);
        double h;
        if (n % 2 == 0)
          h = (y == 0 || y == n / 2) ? 1.0 : (y < n / 2 ? 2.0 : 0.0);
        else
          h = y == 0 ? 1.0 : (y < (n + 1) / 2 ? 2.0 : 0.0);
        const double2 Yc = make_double2(__dmul_rn(X.x, h), __dmul_rn(X.y, -h));
        o = cmul_ra(cy, Yc);
      }
      dst[y] = o;
    } else if (y < n) {  // z = c conj(v) / (M n); |z|
      const double2 conv = make_double2(__dmul_rn(v.x, row.inv_env), __dmul_rn(v.y, -row.inv_env));
      const double2 z = cmul_ra(c[y], conv);
      p.amp[row.out + y] = (float)sqrt(__fma_rn(z.x, z.x, __dmul_rn(z.y, z.y)));
    }
  }
}

}  // namespace

int hilbert_groups(int m, int L[3]) {
  const int G = m <= 22 ? 2 : 3;
  for (int g = 0; g < G; ++g) L[g] = (m + G - 1 - g) / G;  // the larger groups first, each <= 11 bits
  if (G == 2) L[2] = 0;
  return G;
}

long hilbert_items(int m) { return (1L << m) >> kLogE; }

cudaError_t hilbert_varlen_launch(const HilBatch& b, cudaStream_t st) {
  MMF_SMEM_ONCE(hilbert_group_kernel, kE * 16);
  hilbert_chirp_kernel<<<(unsigned)b.chirp_items, 256, 0, st>>>(b.tab, b.chirp_first, b.n_tab, b.s);
  hilbert_twiddle_kernel<<<(unsigned)(((1L << (b.mw - 1)) + 255) / 256), 256, 0, st>>>(1L << (b.mw - 1), b.s + b.w);
  count_launch(2);
  for (int T = 0; T < 5; ++T)
    for (int g = 0; g < b.G; ++g) {
      // rows are ordered three-group rows first: the third group's launch takes only those
      const bool tab = T == 0;
      const long n_rows = g < 2 ? (tab ? b.n_tab : b.n_clip) : (tab ? b.n_tab3 : b.n_clip3);
      if (n_rows == 0) continue;
      const unsigned* first = tab ? b.tab_first : b.clip_first;
      const long items = tab ? (g < 2 ? b.tab_items : b.tab_items3) : (g < 2 ? b.clip_items : b.clip_items3);
      const HilPass p{tab ? b.tab : b.clip, first, n_rows, T, g, b.x, b.pcm16, b.s, b.s + b.w, b.mw, b.amp};
      hilbert_group_kernel<<<(unsigned)items, kThreads, kE * 16, st>>>(p);
      count_launch();
    }
  return cudaGetLastError();
}

}  // namespace mmf
