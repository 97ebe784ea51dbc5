// K4 (chunk-parallel) and the fused K4+K5+K4 "change" kernel.
//
//  * sosfiltfilt_par_kernel: scipy.signal.sosfiltfilt for independent rows whose
//    odd-extended length fits in shared memory; one warp per row (sos_par.cuh).
//  * change_fused_kernel: everything after the MFCC in get_MFCCS_change
//    (script/mfcc.py:393-425) for one clip per CTA: zero-phase Butterworth of every
//    kept coefficient row (one warp per row, rows stay in shared memory),
//    derivative + norm over rows (script/mfcc.py:405-415), and the zero-phase
//    output filter of the resulting curve (script/mfcc.py:417-425) -- the
//    float64 intermediates (96 KB per 10 s clip) never touch HBM.
#include <algorithm>
#include <cfloat>
#include <cstring>
#include <vector>

#include "mmf_internal.h"
#include "sos_par.cuh"

namespace mmf {

// ---------------------------------------------------------------------------
// host: chunk geometry and the zero-input transition matrices
// ---------------------------------------------------------------------------
static void host_sos_step(const SosPar& a, double v, double* z) {
  for (int s = 0; s < a.ns; ++s) {
    const double out = std::fma(a.sos[s][0], v, z[2 * s]);
    z[2 * s] = std::fma(a.sos[s][1], v, std::fma(-a.sos[s][4], out, z[2 * s + 1]));
    z[2 * s + 1] = std::fma(a.sos[s][2], v, -a.sos[s][5] * out);
    v = out;
  }
}

static bool sos_par_fill_cl(const SosArgs& src, int cl, SosPar* out) {
  if (src.n_sections < 1 || src.n_sections > kParMaxSections) return false;
  std::memset(out, 0, sizeof(*out));
  out->ns = src.n_sections;
  out->padlen = src.padlen;
  out->CL = cl;
  for (int s = 0; s < src.n_sections; ++s) {
    for (int k = 0; k < 6; ++k) out->sos[s][k] = src.sos[s][k];
    out->zi[s][0] = src.zi[s][0];
    out->zi[s][1] = src.zi[s][1];
  }
  const int D = 2 * src.n_sections;
  // zero-input transition over one chunk (cl samples), column by column ...
  for (int c = 0; c < D; ++c) {
    double z[2 * kParMaxSections] = {0};
    z[c] = 1.0;
    for (int i = 0; i < cl; ++i) host_sos_step(*out, 0.0, z);
    for (int r = 0; r < D; ++r) out->mpow[0][r][c] = z[r];
  }
  // ... and over 2, 4, 8, 16 chunks and the whole super-block (32 chunks) by repeated squaring
  auto square = [&](const double (*a)[2 * kParMaxSections], double (*m)[2 * kParMaxSections]) {
    for (int r = 0; r < D; ++r)
      for (int c = 0; c < D; ++c) {
        double acc = 0.0;
        for (int k = 0; k < D; ++k) acc = std::fma(a[r][k], a[k][c], acc);
        m[r][c] = acc;
      }
  };
  for (int jj = 1; jj < 5; ++jj) square(out->mpow[jj - 1], out->mpow[jj]);
  square(out->mpow[4], out->msb);
  return true;
}

// the tables depend only on (cascade, chunk length): keep the last few per thread (a variable-length batch uses one
// per odd chunk length of its clips, up to 96 per cascade)
static bool sos_par_cached(const SosArgs& src, int cl, SosPar* out) {
  struct Entry {
    SosArgs key;
    int cl;
    SosPar par;
  };
  static thread_local std::vector<Entry> cache;
  for (const Entry& e : cache)
    if (e.cl == cl && std::memcmp(&e.key, &src, sizeof(SosArgs)) == 0) {
      *out = e.par;
      return true;
    }
  if (!sos_par_fill_cl(src, cl, out)) return false;
  if (cache.size() >= 256) cache.erase(cache.begin());
  Entry e;
  std::memcpy(&e.key, &src, sizeof(SosArgs));
  e.cl = cl;
  e.par = *out;
  cache.push_back(e);
  return true;
}

int sos_par_chunk(const SosArgs& src, long T) {
  const long L = T + 2L * src.padlen;
  if (L > 32L * kSosParMaxChunk) return -1;
  return (int)((L + 31) / 32) | 1;
}

bool sos_par_fill(const SosArgs& src, long T, SosPar* out) {
  const int cl = sos_par_chunk(src, T);
  return cl > 0 && sos_par_cached(src, cl, out);
}

// ---------------------------------------------------------------------------
// generic rows
// ---------------------------------------------------------------------------
constexpr int kParWarps = 4;
constexpr int kFusedPerThread = 9;
constexpr int kFusedMaxWarps = 12;  // 384 threads, <= 85 registers: two CTAs per SM

// VL (variable-length batch): row r is clip vl.clips[r] at x + clip * x_row_stride (packed: at x + vl.off[clip], and
// so is its output row in y) with its own frame count and cascade tables (vl.pidx[clip].y); a warp's buffer is
// `s_stride` doubles, the largest 32 * CL of the launch.
template <typename TIn, int NS, bool VL>
__global__ void __launch_bounds__(kParWarps * 32)
    sosfiltfilt_par_kernel(const TIn* __restrict__ x, long rows, int T, long x_row_stride, int group_rows,
                           long group_stride, const __grid_constant__ SosPar a_, double* __restrict__ y,
                           long y_row_stride, const __grid_constant__ FusedVarlen vl, int s_stride) {
  extern __shared__ __align__(16) double sm_par[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  long row = (long)blockIdx.x * kParWarps + warp;
  if (row >= rows) return;
  if (VL) {
    row = vl.clips[row];
    T = vl.T[row];
  }
  const SosPar& a = VL ? vl.pars[vl.pidx[row].y] : a_;
  const int S = 32 * a.CL, p = a.padlen, L = T + 2 * p;
  double* buf = sm_par + (size_t)warp * s_stride;
  const long g = row / group_rows, gi = row - g * group_rows;
  const bool packed = VL && vl.off != nullptr;
  const long xo = packed ? vl.off[row] : g * group_stride + gi * x_row_stride;
  double* dst = y + (packed ? xo : row * y_row_stride);
  warp_load_odd_ext<TIn>(x + xo, T, p, buf, S, lane);
  const SosRegs<NS> c(a);
  warp_sosfiltfilt<NS>(buf, L, a, c, lane);
  for (int t = lane; t < T; t += 32) dst[t] = buf[p + t];
}

template <typename TIn, int NS>
static cudaError_t par_launch_ns(const TIn* x, long rows, long T, long xs, int group_rows, long group_stride,
                                 const SosPar& a, double* y, long ys, cudaStream_t st) {
  const unsigned grid = (unsigned)((rows + kParWarps - 1) / kParWarps);
  const size_t smem = (size_t)kParWarps * 32 * a.CL * sizeof(double);
  auto kfn = sosfiltfilt_par_kernel<TIn, NS, false>;
  MMF_SMEM_ONCE(kfn, 200 * 1024);
  kfn<<<grid, kParWarps * 32, smem, st>>>(x, rows, (int)T, xs, group_rows, group_stride, a, y, ys, FusedVarlen{},
                                          32 * a.CL);
  count_launch();
  return cudaGetLastError();
}

template <typename TIn, int NS>
static cudaError_t par_varlen_ns(const TIn* x, long rows, long pitch, const SosPar& amax, const FusedVarlen& vl,
                                 double* y, cudaStream_t st) {
  const unsigned grid = (unsigned)((rows + kParWarps - 1) / kParWarps);
  const size_t smem = (size_t)kParWarps * 32 * amax.CL * sizeof(double);
  auto kfn = sosfiltfilt_par_kernel<TIn, NS, true>;
  MMF_SMEM_ONCE(kfn, 200 * 1024);
  kfn<<<grid, kParWarps * 32, smem, st>>>(x, rows, (int)pitch, pitch, 1, pitch, amax, y, pitch, vl, 32 * amax.CL);
  count_launch();
  return cudaGetLastError();
}

template <typename TIn>
static cudaError_t par_varlen_t(const TIn* x, long rows, long pitch, const SosPar& amax, const FusedVarlen& vl,
                                double* y, cudaStream_t st) {
  switch (amax.ns) {
    case 1: return par_varlen_ns<TIn, 1>(x, rows, pitch, amax, vl, y, st);
    case 2: return par_varlen_ns<TIn, 2>(x, rows, pitch, amax, vl, y, st);
    case 3: return par_varlen_ns<TIn, 3>(x, rows, pitch, amax, vl, y, st);
    case 4: return par_varlen_ns<TIn, 4>(x, rows, pitch, amax, vl, y, st);
    default: return cudaErrorInvalidValue;
  }
}

// x_is_f32: float32 rows (the RMS envelope), odd-extended in float32 as the single-row call extends them
cudaError_t sosfiltfilt_par_varlen_launch(const void* x, int x_is_f32, long rows, long pitch, const SosPar& amax,
                                          const FusedVarlen& vl, double* y, cudaStream_t st) {
  if (x_is_f32) return par_varlen_t<float>((const float*)x, rows, pitch, amax, vl, y, st);
  return par_varlen_t<double>((const double*)x, rows, pitch, amax, vl, y, st);
}

template <typename TIn>
static cudaError_t par_launch_t(const TIn* x, long rows, long T, long xs, int group_rows, long group_stride,
                                const SosPar& a, double* y, long ys, cudaStream_t st) {
  switch (a.ns) {
    case 1: return par_launch_ns<TIn, 1>(x, rows, T, xs, group_rows, group_stride, a, y, ys, st);
    case 2: return par_launch_ns<TIn, 2>(x, rows, T, xs, group_rows, group_stride, a, y, ys, st);
    case 3: return par_launch_ns<TIn, 3>(x, rows, T, xs, group_rows, group_stride, a, y, ys, st);
    case 4: return par_launch_ns<TIn, 4>(x, rows, T, xs, group_rows, group_stride, a, y, ys, st);
    default: return cudaErrorInvalidValue;
  }
}

cudaError_t sosfiltfilt_par_launch(const void* x, int x_is_f32, long rows, long T, long xs, int group_rows,
                                   long group_stride, const SosPar& a, double* y, long ys, cudaStream_t st) {
  if (x_is_f32) return par_launch_t<float>((const float*)x, rows, T, xs, group_rows, group_stride, a, y, ys, st);
  return par_launch_t<double>((const double*)x, rows, T, xs, group_rows, group_stride, a, y, ys, st);
}

// ---------------------------------------------------------------------------
// long rows (e.g. the 360 001-frame trajectory of a one-hour recording): the row is cut into
// super-blocks of 32 * CL samples, one warp each, and the state is carried across super-blocks
// the same way it is carried across the lanes of a warp:
//   1. STATE : every super-block's end state from a zero initial state (parallel),
//   2. CARRY : s_in[b+1] = M_sb * s_in[b] + e0[b] along each row (one thread per row, n_sb steps),
//   3. APPLY : every super-block again from its true initial state, writing the output (parallel);
// once forward over the odd-extended input into a scratch row, once backward over that.
// ---------------------------------------------------------------------------
constexpr int kLongCL = 33;
constexpr int kLongWarps = 4;

template <typename TIn>
__device__ __forceinline__ double odd_ext_elem(const TIn* __restrict__ xr, long T, int p, long i) {
  const TIn two = (TIn)2;
  if (i < p) return (double)(TIn)(two * xr[0] - xr[p - i]);
  if (i < p + T) return (double)xr[i - p];
  return (double)(TIn)(two * xr[T - 1] - xr[T - 2 - (i - p - T)]);
}

template <typename TIn, int NS, bool BWD, bool APPLY>
__global__ void __launch_bounds__(kLongWarps * 32)
    sos_long_kernel(const TIn* __restrict__ x, long x_row_stride, int group_rows, long group_stride,
                    const double* __restrict__ fwd_in, long rows, long T, long n_sb, const __grid_constant__ SosPar a,
                    const double* __restrict__ s_in, double* __restrict__ e0, double* __restrict__ fwd_out,
                    double* __restrict__ y, long y_row_stride) {
  extern __shared__ __align__(16) double sm_long[];
  constexpr int D = 2 * NS;
  constexpr int S = 32 * kLongCL;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long unit = (long)blockIdx.x * kLongWarps + warp;
  if (unit >= rows * n_sb) return;
  const long row = unit / n_sb, sb = unit - row * n_sb;
  const int p = a.padlen;
  const long L = T + 2L * p;
  double* buf = sm_long + (size_t)warp * S;
  const long i0 = sb * S;  // first processing index of this super-block
  const long g = row / group_rows, gi = row - g * group_rows;
  const TIn* xr = x + g * group_stride + gi * x_row_stride;
  const double* fr = fwd_in + row * L;
  for (int j = lane; j < S; j += 32) {
    const long i = i0 + j;
    double v = 0.0;
    if (i < L) v = BWD ? fr[L - 1 - i] : odd_ext_elem<TIn>(xr, T, p, i);
    buf[j] = v;
  }
  __syncwarp();
  const SosRegs<NS> c(a);
  const int n_here = (int)min((long)S, L - i0);
  double s0[D], z[D];
  if (APPLY) {
#pragma unroll
    for (int i = 0; i < D; ++i) s0[i] = s_in[unit * D + i];
    warp_sos_core<NS, false, true>(buf, n_here, a, c, lane, s0, z);
    for (int j = lane; j < n_here; j += 32) {
      const long i = i0 + j;
      if (BWD) {
        const long e = L - 1 - i;
        if (e >= p && e < p + T) y[row * y_row_stride + (e - p)] = buf[j];
      } else {
        fwd_out[row * L + i] = buf[j];
      }
    }
  } else {
#pragma unroll
    for (int i = 0; i < D; ++i) s0[i] = 0.0;
    warp_sos_core<NS, false, false>(buf, n_here, a, c, lane, s0, z);
    if (lane == 31) {
#pragma unroll
      for (int i = 0; i < D; ++i) e0[unit * D + i] = z[i];
    }
  }
}

template <typename TIn, int NS, bool BWD>
__global__ void sos_long_carry_kernel(const TIn* __restrict__ x, long x_row_stride, int group_rows, long group_stride,
                                      const double* __restrict__ fwd_in, long rows, long T, long n_sb,
                                      const __grid_constant__ SosPar a, const double* __restrict__ e0,
                                      double* __restrict__ s_in) {
  constexpr int D = 2 * NS;
  const long row = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= rows) return;
  const int p = a.padlen;
  const long L = T + 2L * p;
  const long g = row / group_rows, gi = row - g * group_rows;
  const double u0 = BWD ? fwd_in[row * L + L - 1] : odd_ext_elem<TIn>(x + g * group_stride + gi * x_row_stride, T, p, 0);
  double s[D];
#pragma unroll
  for (int q = 0; q < NS; ++q) {
    s[2 * q] = a.zi[q][0] * u0;
    s[2 * q + 1] = a.zi[q][1] * u0;
  }
  for (long b = 0; b < n_sb; ++b) {
    const long unit = row * n_sb + b;
    double nx[D];
#pragma unroll
    for (int r = 0; r < D; ++r) {
      s_in[unit * D + r] = s[r];
      double acc = e0[unit * D + r];
#pragma unroll
      for (int i = 0; i < D; ++i) acc = fma(a.msb[r][i], s[i], acc);
      nx[r] = acc;
    }
#pragma unroll
    for (int r = 0; r < D; ++r) s[r] = nx[r];
  }
}

template <typename TIn, int NS>
static cudaError_t long_launch_ns(const TIn* x, long rows, long T, long xs, int group_rows, long group_stride,
                                  const SosPar& a, double* y, long ys, cudaStream_t st) {
  constexpr int D = 2 * NS;
  const long S = 32L * kLongCL, L = T + 2L * a.padlen, n_sb = (L + S - 1) / S;
  const long units = rows * n_sb;
  double *fwd = nullptr, *e0 = nullptr, *sin_ = nullptr;
  cudaError_t e;
  if ((e = cudaMallocAsync((void**)&fwd, (size_t)rows * L * 8, st)) != cudaSuccess) return e;
  if ((e = cudaMallocAsync((void**)&e0, (size_t)units * D * 8, st)) != cudaSuccess) {
    cudaFreeAsync(fwd, st);
    return e;
  }
  if ((e = cudaMallocAsync((void**)&sin_, (size_t)units * D * 8, st)) != cudaSuccess) {
    cudaFreeAsync(fwd, st);
    cudaFreeAsync(e0, st);
    return e;
  }
  const unsigned grid = (unsigned)((units + kLongWarps - 1) / kLongWarps);
  const unsigned cgrid = (unsigned)((rows + 63) / 64);
  const size_t smem = (size_t)kLongWarps * S * 8;
  sos_long_kernel<TIn, NS, false, false><<<grid, kLongWarps * 32, smem, st>>>(x, xs, group_rows, group_stride, fwd, rows,
                                                                            T, n_sb, a, sin_, e0, fwd, y, ys);
  sos_long_carry_kernel<TIn, NS, false><<<cgrid, 64, 0, st>>>(x, xs, group_rows, group_stride, fwd, rows, T, n_sb, a, e0,
                                                              sin_);
  sos_long_kernel<TIn, NS, false, true><<<grid, kLongWarps * 32, smem, st>>>(x, xs, group_rows, group_stride, fwd, rows,
                                                                           T, n_sb, a, sin_, e0, fwd, y, ys);
  sos_long_kernel<TIn, NS, true, false><<<grid, kLongWarps * 32, smem, st>>>(x, xs, group_rows, group_stride, fwd, rows,
                                                                           T, n_sb, a, sin_, e0, fwd, y, ys);
  sos_long_carry_kernel<TIn, NS, true><<<cgrid, 64, 0, st>>>(x, xs, group_rows, group_stride, fwd, rows, T, n_sb, a, e0,
                                                             sin_);
  sos_long_kernel<TIn, NS, true, true><<<grid, kLongWarps * 32, smem, st>>>(x, xs, group_rows, group_stride, fwd, rows, T,
                                                                          n_sb, a, sin_, e0, fwd, y, ys);
  count_launch(6);
  e = cudaGetLastError();
  cudaFreeAsync(fwd, st);
  cudaFreeAsync(e0, st);
  cudaFreeAsync(sin_, st);
  return e;
}

template <typename TIn>
static cudaError_t long_launch_t(const TIn* x, long rows, long T, long xs, int group_rows, long group_stride,
                                 const SosPar& a, double* y, long ys, cudaStream_t st) {
  switch (a.ns) {
    case 1: return long_launch_ns<TIn, 1>(x, rows, T, xs, group_rows, group_stride, a, y, ys, st);
    case 2: return long_launch_ns<TIn, 2>(x, rows, T, xs, group_rows, group_stride, a, y, ys, st);
    case 3: return long_launch_ns<TIn, 3>(x, rows, T, xs, group_rows, group_stride, a, y, ys, st);
    case 4: return long_launch_ns<TIn, 4>(x, rows, T, xs, group_rows, group_stride, a, y, ys, st);
    default: return cudaErrorInvalidValue;
  }
}

bool sos_long_supported(const SosArgs& a, long rows, long T) {
  const long L = T + 2L * a.padlen;
  return a.n_sections >= 1 && a.n_sections <= kParMaxSections && L > 32L * kLongCL &&
         rows * ((L + 32L * kLongCL - 1) / (32L * kLongCL)) < 0x7fffffffL * kLongWarps;
}

cudaError_t sosfiltfilt_long_launch(const void* x, int x_is_f32, long rows, long T, long xs, int group_rows,
                                    long group_stride, const SosArgs& src, double* y, long ys, cudaStream_t st) {
  SosPar a;
  if (!sos_par_cached(src, kLongCL, &a)) return cudaErrorInvalidValue;
  if (x_is_f32) return long_launch_t<float>((const float*)x, rows, T, xs, group_rows, group_stride, a, y, ys, st);
  return long_launch_t<double>((const double*)x, rows, T, xs, group_rows, group_stride, a, y, ys, st);
}

// ---------------------------------------------------------------------------
// fused per-clip kernel
// ---------------------------------------------------------------------------
// K3 folded into the per-clip kernel: clamp + DCT-II of this clip's log-mel columns straight into the
// float64 row buffers (and to HBM as float32 MFCC / delta when the caller wants them).  Same FMA order
// per coefficient as mfcc_kernel (post_kernels.cu), so the MFCCs are bit-identical to the unfused path.
constexpr int kFusedDepth = 8;  // log-mel rows in flight per thread (16 measured slower)
__device__ __forceinline__ float fused_key_to_float(int k) { return __int_as_float(k >= 0 ? k : k ^ 0x7FFFFFFF); }

__device__ __forceinline__ void fused_mfcc_phase(const FusedMfccArgs& m, long clip, int n_mfcc, int first, int T,
                                                 int pitch, int S, int p, double* rowbuf, float* s_dct) {
  const int tid = threadIdx.x, nthr = blockDim.x, lane = tid & 31;
  const int n_mels = m.n_mels;
  for (int i = tid; i < n_mels * kFusedNC; i += nthr) {
    const int mm = i / kFusedNC, j = i - mm * kFusedNC;
    s_dct[i] = m.dct_pad[mm * m.dct_pitch + j];
  }
  __syncthreads();
  const float thr = m.top_db >= 0.0f ? fused_key_to_float(m.clipmax[clip]) - m.top_db : -FLT_MAX;
  // a warp takes 32 consecutive frames; with delta wanted the outer two are a halo (recomputed by the
  // neighbouring tile) so that t-1 / t+1 come from lane shuffles instead of shared memory
  const int halo = m.delta_out != nullptr ? 1 : 0;
  const int width = 32 - 2 * halo;
  const int n_tiles = (T + width - 1) / width;
  for (int tile = tid >> 5; tile < n_tiles; tile += nthr >> 5) {
    const int t = tile * width - halo + lane;
    const bool valid = t >= 0 && t < T;
    const bool own = valid && lane >= halo && lane < 32 - halo;
    float acc[kFusedNC];
#pragma unroll
    for (int j = 0; j < kFusedNC; ++j) acc[j] = 0.0f;
    if (valid) {
      float* col = m.logmel + (size_t)clip * n_mels * pitch + t;
      float cur[kFusedDepth], nxt[kFusedDepth];
#pragma unroll
      for (int u = 0; u < kFusedDepth; ++u) cur[u] = (u < n_mels) ? __ldcs(col + (size_t)u * pitch) : 0.0f;
      for (int m0 = 0; m0 < n_mels; m0 += kFusedDepth) {
#pragma unroll
        for (int u = 0; u < kFusedDepth; ++u)
          nxt[u] = (m0 + kFusedDepth + u < n_mels) ? __ldcs(col + (size_t)(m0 + kFusedDepth + u) * pitch) : 0.0f;
#pragma unroll
        for (int u = 0; u < kFusedDepth; ++u) {
          const int mm = m0 + u;
          if (mm < n_mels) {
            const float x = fmaxf(cur[u], thr);
            if (m.clamp_in_place && own) col[(size_t)mm * pitch] = x;
            const float4* d4 = reinterpret_cast<const float4*>(s_dct + mm * kFusedNC);
#pragma unroll
            for (int j4 = 0; j4 < kFusedNC / 4; ++j4) {
              const float4 d = d4[j4];
              acc[4 * j4 + 0] = fmaf(d.x, x, acc[4 * j4 + 0]);
              acc[4 * j4 + 1] = fmaf(d.y, x, acc[4 * j4 + 1]);
              acc[4 * j4 + 2] = fmaf(d.z, x, acc[4 * j4 + 2]);
              acc[4 * j4 + 3] = fmaf(d.w, x, acc[4 * j4 + 3]);
            }
          }
        }
#pragma unroll
        for (int u = 0; u < kFusedDepth; ++u) cur[u] = nxt[u];
      }
    }
    if (own) {
      float* dst = m.mfcc_out ? m.mfcc_out + (size_t)clip * n_mfcc * pitch + t : nullptr;
#pragma unroll
      for (int j = 0; j < kFusedNC; ++j) {
        if (j < n_mfcc) {
          if (dst) dst[(size_t)j * pitch] = acc[j];
          if (j >= first) rowbuf[(size_t)(j - first) * S + p + t] = (double)acc[j];
        }
      }
    }
    if (halo) {
      // delta = np.gradient along time in float32 (calc.py:642-645); shuffles stay outside any
      // lane-dependent branch
      float* dst = m.delta_out + (size_t)clip * n_mfcc * pitch + t;
#pragma unroll
      for (int j = 0; j < kFusedNC; ++j) {
        if (j < n_mfcc) {
          const float cp = __shfl_down_sync(0xffffffffu, acc[j], 1);
          const float cm = __shfl_up_sync(0xffffffffu, acc[j], 1);
          float d;
          if (T == 1) d = 0.0f;
          else if (t == 0) d = cp - acc[j];
          else if (t == T - 1) d = acc[j] - cm;
          else d = (cp - cm) / 2.0f;
          if (own) dst[(size_t)j * pitch] = d;
        }
      }
    }
  }
  __syncthreads();
}

// VL (variable-length batch): CTA b takes clip vl.clips[b] with its own frame count and cascade tables; `T` is then
// the row pitch of every input and output.
template <int NS1, int NS2, bool FROM_LM, bool VL>
__global__ void __launch_bounds__(kFusedMaxWarps * 32, 2)
    change_fused_kernel(const float* __restrict__ mfcc, int n_mfcc, int first, int rows, int T, int method,
                        const __grid_constant__ SosPar a1_, const __grid_constant__ SosPar a2_, int out_kind,
                        double* __restrict__ tot, const __grid_constant__ FusedMfccArgs lm, int sm_doubles,
                        const __grid_constant__ FusedVarlen vl) {
  extern __shared__ __align__(16) double sm_fused[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
  const long clip = VL ? vl.clips[blockIdx.x] : blockIdx.x;
  const int pitch = T;
  if (VL) T = vl.T[clip];
  const SosPar& a1 = VL ? vl.pars[vl.pidx[clip].x] : a1_;
  const SosPar& a2 = VL ? vl.pars[vl.pidx[clip].y] : a2_;
  const int S = 32 * a1.CL, p = a1.padlen, L = T + 2 * p;
  if (FROM_LM) {
    float* s_dct = reinterpret_cast<float*>(sm_fused + sm_doubles);
    fused_mfcc_phase(lm, clip, n_mfcc, first, T, pitch, S, p, sm_fused, s_dct);
  }
  // 1. zero-phase Butterworth of every kept coefficient row, in place in shared memory
  {
    const SosRegs<NS1> c1(a1);
    for (int r = warp; r < rows; r += nwarps) {
      double* buf = sm_fused + (size_t)r * S;
      if (FROM_LM) warp_odd_ext_staged<float>(buf, T, p, S, lane);
      else warp_load_odd_ext<float>(mfcc + ((size_t)clip * n_mfcc + first + r) * pitch, T, p, buf, S, lane);
      warp_sosfiltfilt<NS1>(buf, L, a1, c1, lane);
    }
  }
  __syncthreads();
  // 2. derivative along time and norm over rows (script/mfcc.py:405-415)
  constexpr int kPerThread = kFusedPerThread;  // the launcher guarantees T <= blockDim * kPerThread
  double raw[kPerThread];
#pragma unroll
  for (int q = 0; q < kPerThread; ++q) {
    const int t = tid + q * blockDim.x;
    double s = 0.0;
    if (t < T) {
      for (int r = 0; r < rows; ++r) {
        const double* f = sm_fused + (size_t)r * S + p;
        double d;
        if (T == 1) {
          d = 0.0;
        } else if (t == 0) {
          d = (method == 0 || T < 3) ? f[1] - f[0] : (-3.0 * f[0] + 4.0 * f[1] - f[2]) / 2.0;
        } else if (t == T - 1) {
          d = (method == 0 || T < 3) ? f[T - 1] - f[T - 2] : (3.0 * f[T - 1] - 4.0 * f[T - 2] + f[T - 3]) / 2.0;
        } else {
          d = (f[t + 1] - f[t - 1]) / 2.0;
        }
        s += d * d;
      }
    }
    raw[q] = sqrt(s) / (double)rows;
  }
  double* dst = tot + (size_t)clip * pitch;
  if (out_kind != 0) {
#pragma unroll
    for (int q = 0; q < kPerThread; ++q) {
      const int t = tid + q * blockDim.x;
      if (t < T) dst[t] = raw[q];
    }
    return;
  }
  __syncthreads();  // every row has been read: row 0's buffer becomes the curve's buffer
  // 3. output filter of the curve (script/mfcc.py:417-425); the two cascades may differ in padlen
  const int p2 = a2.padlen, L2 = T + 2 * p2, S2 = 32 * a2.CL;
  double* cbuf = sm_fused;
#pragma unroll
  for (int q = 0; q < kPerThread; ++q) {
    const int t = tid + q * blockDim.x;
    if (t < T) cbuf[p2 + t] = raw[q];
  }
  __syncthreads();
  for (int i = tid; i < S2; i += blockDim.x) {
    if (i < p2) {
      cbuf[i] = 2.0 * cbuf[p2] - cbuf[p2 + (p2 - i)];
    } else if (i >= p2 + T) {
      cbuf[i] = i < L2 ? 2.0 * cbuf[p2 + T - 1] - cbuf[p2 + T - 2 - (i - p2 - T)] : 0.0;
    }
  }
  __syncthreads();
  if (warp == 0) {
    const SosRegs<NS2> c2(a2);
    warp_sosfiltfilt<NS2>(cbuf, L2, a2, c2, lane);
  }
  __syncthreads();
  for (int t = tid; t < T; t += blockDim.x) dst[t] = cbuf[p2 + t];
}

static size_t fused_row_doubles(const SosPar& a1, const SosPar* a2, int rows) {
  size_t doubles = (size_t)rows * 32 * a1.CL;
  if (a2) doubles = std::max(doubles, (size_t)32 * a2->CL);
  return doubles;
}

bool change_fused_supported(const SosPar& a1, const SosPar* a2, bool split_out, int rows, long T, size_t* smem_out) {
  if (rows < 1 || T < 1 || T > (long)kFusedMaxWarps * 32 * kFusedPerThread) return false;
  // equal section counts (the reference's default: outFilter None reuses the row filter, 'iir' uses the same order)
  // get an instantiation; a kernel that leaves the output filter to its own launch instantiates the row filter only
  if (a2 && !split_out && a2->ns != a1.ns) return false;
  const size_t smem = fused_row_doubles(a1, a2, rows) * sizeof(double);
  if (smem > 220 * 1024) return false;
  if (smem_out) *smem_out = smem;
  return true;
}

// with the MFCC stage folded in: + the DCT table
bool change_fused_lm_supported(const SosPar& a1, const SosPar* a2, bool split_out, int n_mfcc, int n_mels, int first,
                               int rows, long T, size_t* smem_out) {
  size_t base = 0;
  if (n_mfcc > kFusedNC || !change_fused_supported(a1, a2, split_out, rows, T, &base)) return false;
  const size_t smem = base + (size_t)n_mels * kFusedNC * sizeof(float);
  if (smem > 220 * 1024) return false;
  if (smem_out) *smem_out = smem;
  return true;
}

template <int NS1, int NS2, bool VL>
static cudaError_t fused_launch_cl(const float* mfcc, long n_clips, int n_mfcc, int first, int rows, long T,
                                   int method, const SosPar& a1, const SosPar& a2, int out_kind, double* tot,
                                   size_t smem, const FusedMfccArgs* lm, cudaStream_t st, const FusedVarlen& vl) {
  // >= ceil(T / (32*kFusedPerThread)) warps for the derivative phase, one per row if possible
  int warps = std::min(kFusedMaxWarps, std::max(rows, (int)((T + 32 * kFusedPerThread - 1) / (32 * kFusedPerThread))));
  const int sm_doubles = (int)fused_row_doubles(a1, out_kind == 0 ? &a2 : nullptr, rows);
  if (lm) {
    // the DCT phase streams the clip's log-mel columns: it wants every thread the CTA may have
    warps = kFusedMaxWarps;
    auto kfn = change_fused_kernel<NS1, NS2, true, VL>;
    MMF_SMEM_ONCE(kfn, 220 * 1024);
    kfn<<<(unsigned)n_clips, warps * 32, smem, st>>>(nullptr, n_mfcc, first, rows, (int)T, method, a1, a2, out_kind,
                                                     tot, *lm, sm_doubles, vl);
  } else {
    auto kfn = change_fused_kernel<NS1, NS2, false, VL>;
    MMF_SMEM_ONCE(kfn, 220 * 1024);
    kfn<<<(unsigned)n_clips, warps * 32, smem, st>>>(mfcc, n_mfcc, first, rows, (int)T, method, a1, a2, out_kind,
                                                     tot, FusedMfccArgs{}, sm_doubles, vl);
  }
  count_launch();
  return cudaGetLastError();
}

cudaError_t change_fused_launch(const float* mfcc, long n_clips, int n_mfcc, int first, int rows, long T, int method,
                                const SosPar& a1, const SosPar& a2, int out_kind, double* tot, size_t smem,
                                const FusedMfccArgs* lm, cudaStream_t st, const FusedVarlen* vl) {
  // one instantiation per equal section count (change_fused_supported)
  const int k = a1.ns * 10 + (out_kind == 0 ? a2.ns : a1.ns);
  switch (k) {
#define MMF_FUSED_CASE(A, B)                                                                                          \
  case A * 10 + B:                                                                                                    \
    return vl ? fused_launch_cl<A, B, true>(mfcc, n_clips, n_mfcc, first, rows, T, method, a1, a2, out_kind, tot, smem, \
                                            lm, st, *vl)                                                              \
              : fused_launch_cl<A, B, false>(mfcc, n_clips, n_mfcc, first, rows, T, method, a1, a2, out_kind, tot,    \
                                             smem, lm, st, FusedVarlen{});
    MMF_FUSED_CASE(1, 1)
    MMF_FUSED_CASE(2, 2)
    MMF_FUSED_CASE(3, 3)
    MMF_FUSED_CASE(4, 4)
#undef MMF_FUSED_CASE
    default: return cudaErrorNotSupported;
  }
}

}  // namespace mmf
