// Internal declarations shared by the kernels and the C ABI (not installed).
#pragma once
#include <cuda.h>
#include <cudaTypedefs.h>
#include <cuda_runtime.h>

#include <cstddef>
#include <cstdint>
#include <string>
#include <vector>

#include "../../include/mmf.h"

namespace mmf {

// ---- a variable-length batch (mmf_mfcc_change_varlen): device arrays built per call.  Clip i has len[i] samples
// and T[i] frames; T[i] = 0 marks a clip the launch skips (it takes the single-clip path).  K1 walks a compacted list
// of work units (128-frame blocks or TF-frame tiles): clip i owns units [first[i], first[i + 1]).  Output rows are
// `pitch` (the longest clip's T) frames apart.
struct Varlen {
  const long* len;
  const int* T;
  const unsigned* first;
  long n_units;
  int pitch;
};

// ---- arguments of the fused STFT/mel kernel (passed by value)
struct StftArgs {
  const float* pcm;
  long n_samples;
  long clip_stride;
  long n_tiles;
  int tiles_per_clip;
  int T;
  int hop;
  int TF;                // frames per tile (power of two, <= 32, multiple of frames/iteration)
  int span_floats;       // (TF-1)*hop + n_fft + lead + 3 (start rounded down to 4 floats)
  int span_alloc;        // span_floats rounded up to 256-float TMA boxes
  int ppitch;            // power-tile row pitch (floats)
  int pt_bufs;           // power-tile buffers (2 = double buffered, 1 = extra barrier per tile)
  int span_bufs;         // PCM span buffers (2 = prefetch at tile start, 1 = prefetch after the FFT phase)
  int lead;              // samples loaded ahead of the first frame (2 when pre-emphasis is on)
  int use_tma;
  int vec_ok;            // 64-bit shared loads allowed (hop even)
  int split_regs;        // n_fft = 512: shuffle-based split step
  int mel_mma;           // mel projection on the tensor cores (mma.sync TF32 x3) instead of the sparse FP32 walk
  int m_tiles;           // 16-frame MMA row tiles per tile of TF frames (1 or 2)
  int mma_n_pairs;       // non-zero (n-tile, k-tile) blocks of the filterbank
  int mel_tab_bytes;     // shared-memory bytes of the mel tables of the active mode
  const float2* mma_bw;  // [n_pairs][32] B fragments: W[8*k8 + lane%4 (+4)][8*n + lane/4], n-major
  const int* mma_pk8;    // [n_pairs] k-tile of each block
  const int* mma_npair;  // [NT + 1] block range of each n-tile
  const int* mma_tile;   // [NT] first band | bands << 16 of each n-tile (up to 8 consecutive bands)
  int mma_n_tiles;
  const int* mma_units;  // [8][16] (n | m << 8) units of each warp, -1 terminated
  int early_tma;         // single span buffer: prefetch the next tile right after the load phase (extra barrier)
  int debug_skip;        // profiling aid (MMF_DEBUG_SKIP): bit 0 skips the FFT phase, bit 1 the mel phase
  int threads;           // CTA size: 256 (two CTAs per SM) or 512 (one)
  int packed;            // two frames per thread group on packed FP32 instructions (FFMA2/FADD2)
  int n_mels;
  float amin;
  float preemph;
  const float* window;   // [n_fft]
  const float2* tw1;     // [16*TPF]
  const float2* tw2;     // [16*R3]
  const int* seg_start;  // [n_mels + 2]
  const int* band_split; // [257] first band of each mel worker (balanced band groups), padded with n_mels
  const float2* w2;      // [F] (falling, rising) mel weights per bin
  int mel_groups;        // grouped mel walk on the bin-pair tile layout (default) instead of the sparse walk
  int mg_n;              // weight groups of the grouped walk
  const int2* mg_seg;    // [n_mels + 2] (first 4-bin group, first weight group) per segment
  const int2* mg_step;   // [n_mels + 3] (weight groups, tile-pointer step in 8-byte words before the segment)
  const float4* mg_w;    // [2 * mg_n] falling / rising weights of each group
  float* logmel;         // [n_clips, n_mels, T] or null
  int* clipmax;          // [n_clips] float keys or null
  float* power;          // [n_clips, F, T] or null
  int pitch;             // frames per log-mel / power row (T, or the longest clip's T in a variable-length batch)
  const long* vl_len;    // variable-length batch (else null): see Varlen
  const int* vl_T;
  const unsigned* vl_first;
  int vl_clips;
};

struct StftGeometry {
  int tpf, fpi, tw1, tw2, r3, m;
};

bool stft_packed_supported(int n_fft);
int stft_geometry(int n_fft, int packed, int threads, StftGeometry* g);
size_t stft_mel_table_bytes(int n_fft, int n_mels, int mel_mma, int n_pairs, int n_tiles, int mel_groups = 0,
                            int mg_n = 0);
size_t stft_smem_bytes(int n_fft, int span_alloc, int span_bufs, int ppitch, int pt_bufs, int packed,
                       size_t mel_tab_bytes, int threads, int mel_groups = 0);
cudaError_t stft_mel_launch(int n_fft, const CUtensorMap& tmap, const StftArgs& a, int grid, size_t smem,
                            cudaStream_t st);

// ---- K1 with the mel projection as a tcgen05 GEMM over 128-frame blocks (stft_mel_tc.cu; n_fft = 512, <= 112 non-empty bands)
int stft_mel_tc_active_bands(const std::vector<float>& mel, int n_mels, int F);
bool stft_mel_tc_supported(int n_fft, int n_act, int hop, int lead, int packed);
void stft_mel_tc_table(const std::vector<float>& mel, int n_mels, int F, std::vector<uint16_t>& tab);
cudaError_t stft_mel_tc_launch(const CUtensorMap& tmap, int use_tma, const float* pcm, long n_clips, long n_samples,
                               long clip_stride, int T, int hop,
                               int lead, int n_mels, int n_act, float amin, float preemph, const float* window, int win_lo,
                               int win_hi, const float2* tw1, const void* wtab, float* logmel, int* clipmax,
                               int sm_count, cudaStream_t st, const Varlen* vl = nullptr);

// ---- generic n_fft (anything but a power of two in [256, 4096]): FP32 matrix-product DFT (dft_generic.cu)
void dft_generic_table(int n_fft, const std::vector<float>& window, std::vector<float>& tab, int* ld_out);
cudaError_t dft_generic_power_launch(const float* pcm, long n_clips, long n_samples, long clip_stride, int T, int hop,
                                     int n_fft, float preemph, const float* btab, int ld_b, float* power,
                                     cudaStream_t st);
cudaError_t mel_from_power_launch(const float* power, long n_clips, int F, int T, int n_mels, float amin,
                                  const int* seg_start, const float2* w2, float* logmel, int* clipmax,
                                  cudaStream_t st);

// ---- 512-point frames on the tcgen05 tensor cores (tc_fft.cu, MMF_FLAG_TC_FFT)
void tc_fft_tables(std::vector<uint16_t>& btab, std::vector<float>& tw);
bool tc_fft_supported(int n_fft, int hop, float preemph);
cudaError_t tc_fft_power_launch(const float* pcm, long n_clips, long n_samples, long clip_stride, int T, int hop,
                                const float* window, const void* btab, const float2* tw, float* power, int sm_count,
                                cudaStream_t st);

// ---- clamp + DCT-II (+ delta) as a tcgen05 GEMM (mfcc_tc.cu)
bool mfcc_tc_supported(int n_mfcc, int n_mels);
void mfcc_tc_table(const float* dct, int n_mfcc, int n_mels, std::vector<uint16_t>& tab, int* kp_out);
cudaError_t mfcc_tc_launch(const void* btab, int kp, float* logmel, const int* clipmax, long n_clips, long T, int n_mels,
                           int n_mfcc, float top_db, float* mfcc, float* delta, int clamp_in_place, int sm_count,
                           cudaStream_t st);

// ---- K6 routing: the kernel mmf_modspec runs for n_clips clips of T frames and the windows per CTA (wc) it cuts
// each clip's windows into.  One function owns the decision (c_api.cu): mmf_modspec and mmf_modspec_varlen, which
// routes every clip of a ragged batch as its own call would, both take it from here.  n_bands counts band outputs
// actually written (0 without a band output); n_clips only matters through the grid limits.
enum ModPath { kModNone = 0, kModTc, kModClip, kModFast, kModGeneric };
struct ModRoute {
  ModPath path;
  long wc;        // tc / clip: windows per chunk
  long n_chunks;  // tc / clip: chunks per clip
};
ModRoute modspec_route(int win, int hop, int nfft, int n_coef, int n_bands, long T, unsigned flags, long n_clips = 1);
// the chunk sizes behind it: 0 when the kernel does not take the geometry
long modspec_tc_chunk(int win, int hop, int nfft, int n_coef, int n_bands, long T);
long modspec_clip_chunk(int win, int hop, int nfft, int n_coef, int n_bands, long T);

// ---- a variable-length batch of K6 (mmf_modspec_varlen): the launch walks a compacted list of work items, one per
// (clip, chunk of windows) exactly as the clip's own mmf_modspec call cuts it.  Input rows are the launch's T (the row
// pitch) frames apart, output rows its n_win (the most windows of any clip) windows apart.
struct alignas(16) ModItem {
  int clip, w0, wca;  // clip, first window, windows of the chunk
  int n_win;          // windows of the clip
};
struct ModVarlen {
  const ModItem* items;
  long n_items;
  long n_win;  // windows per output row: the most windows of any clip
  int wc_max;  // the most windows of any item: sizes shared memory
};

// ---- modulation spectrum as a tcgen05 GEMM (modspec_tc.cu)
bool modspec_tc_supported(int win, int nfft);
void modspec_tc_table(int win, int nfft, std::vector<uint16_t>& g, int* kp_out);
// wc: modspec_route's chunk size (vl: the batch's items instead)
cudaError_t modspec_tc_launch(const float* mfcc, long n_clips, int n_coef, long T, int win, int hop, int nfft,
                              const void* g, int kp, long wc, float* mag, float* band, const int* lo, const int* hi,
                              int n_bands, int sm_count, cudaStream_t st, const ModVarlen* vl = nullptr);

// ---- post-FFT kernels (post_kernels.cu)
cudaError_t mfcc_launch(const float* dct_pad, int nc_pad, float* logmel, const int* clipmax, long n_clips, long T,
                        int n_mels, int n_mfcc, float top_db, float* mfcc, float* delta, int clamp_in_place,
                        cudaStream_t st, const int* vT = nullptr);

void mfcc_mma_bfrag(const float* dct, int n_mfcc, int n_mels, std::vector<float4>& out);
bool mfcc_mma_supported(int n_mfcc, int n_mels);
cudaError_t mfcc_mma_launch(const float4* bfrag_dev, float* logmel, const int* clipmax, long n_clips, long T, int n_mels,
                            int n_mfcc, float top_db, float* mfcc, float* delta, int clamp_in_place, cudaStream_t st);

struct SosArgs {
  int n_sections;
  int padlen;
  double sos[16][6];
  double zi[16][2];
};
cudaError_t sosfiltfilt_launch(const void* x, int x_is_f32, long rows, long T, long xs, const SosArgs& a, double* y,
                               long ys, cudaStream_t st);
cudaError_t sosfiltfilt_launch_grouped(const void* x, int x_is_f32, long rows, long T, long xs, int group_rows,
                                       long group_stride, const SosArgs& a, double* y, long ys, cudaStream_t st);
// chunk-parallel zero-phase IIR and the fused per-clip change kernel (change_fused.cu)
constexpr int kSosParMaxChunk = 191;  // rows up to 32*191 = 6112 extended samples stay in shared memory
struct SosPar;
bool sos_par_fill(const SosArgs& src, long T, SosPar* out);
cudaError_t sosfiltfilt_par_launch(const void* x, int x_is_f32, long rows, long T, long xs, int group_rows,
                                   long group_stride, const SosPar& a, double* y, long ys, cudaStream_t st);
bool sos_long_supported(const SosArgs& a, long rows, long T);
cudaError_t sosfiltfilt_long_launch(const void* x, int x_is_f32, long rows, long T, long xs, int group_rows,
                                    long group_stride, const SosArgs& a, double* y, long ys, cudaStream_t st);
bool change_fused_supported(const SosPar& a1, const SosPar* a2, int rows, long T, size_t* smem_out);
// K3 folded into the fused kernel (lm != nullptr) takes up to kFusedNC coefficients
constexpr int kFusedNC = 16;
// K3 folded into the fused kernel (lm != nullptr): the clip's MFCC rows go from the DCT straight into
// the float64 row buffers; mfcc_out / delta_out are optional HBM copies for the caller
struct FusedMfccArgs {
  const float* dct_pad;
  int dct_pitch;
  float* logmel;
  const int* clipmax;
  int n_mels;
  float top_db;
  float* mfcc_out;
  float* delta_out;
  int clamp_in_place;
};
bool change_fused_lm_supported(const SosPar& a1, const SosPar* a2, int n_mfcc, int n_mels, int first, int rows,
                               long T, size_t* smem_out);
// variable-length batch of the fused kernel and the batched output filter: launch item b is clip clips[b] with T[clip]
// frames and the cascade tables pars[pidx[clip].x] (row filter) / pars[pidx[clip].y] (output filter); the launch's
// T is the row pitch and its SosPar arguments are the ones with the largest chunk (they size shared memory).  off
// (batched output filter only): packed rows, clip's input and output rows both at off[clip] (null: at clip * pitch)
struct FusedVarlen {
  const int* clips;
  const int* T;
  const SosPar* pars;
  const int2* pidx;
  const long* off = nullptr;
};
cudaError_t change_fused_launch(const float* mfcc, long n_clips, int n_mfcc, int first, int rows, long T, int method,
                                const SosPar& a1, const SosPar& a2, int out_kind, double* tot, size_t smem,
                                const FusedMfccArgs* lm, cudaStream_t st, const FusedVarlen* vl = nullptr);
cudaError_t sosfiltfilt_par_varlen_launch(const void* x, int x_is_f32, long rows, long pitch, const SosPar& amax,
                                          const FusedVarlen& vl, double* y, cudaStream_t st);
cudaError_t varlen_tails_launch(long n_clips, const int* T, int pitch, double* tot, float* logmel, int n_mels,
                                float* mfcc, float* delta, int n_mfcc, cudaStream_t st);
cudaError_t delta_norm_launch(const double* x, long n_clips, int rows, long T, int method, double* tot,
                              cudaStream_t st);
cudaError_t fir_filtfilt_launch(const double* x, long rows, long T, const double* b_dev, int n_taps, double* y,
                                double* work, cudaStream_t st);
cudaError_t stencil_launch(const double* x, long rows, long T, const double* coef_dev, int half, const double* el_dev,
                           const double* er_dev, int n_edge, int n_edge_in, double* y, cudaStream_t st);
cudaError_t modspec_launch(const float* mfcc, long n_clips, int n_coef, long T, int win, int hop, int nfft, float* mag,
                           float* band, const int* band_lo_dev, const int* band_hi_dev, int n_bands, cudaStream_t st);
cudaError_t modspec_tails_launch(long n_clips, const int* n_win, long W, float* mag, int n_coef, int nb, float* band,
                                 int n_bands, cudaStream_t st);
bool modspec_fast_supported(int nfft);
void modspec_geometry(int nfft, StftGeometry* g);
cudaError_t modspec_fast_launch(const float* mfcc, long n_clips, int n_coef, long T, int win, int hop, int nfft,
                                const float* hann, const float2* tw1, const float2* tw2, float* mag, float* band,
                                const int* lo, const int* hi, int n_bands, int sm_count, cudaStream_t st);
// wc: modspec_route's chunk size (vl: the batch's items instead)
cudaError_t modspec_clip_launch(const float* mfcc, long n_clips, int n_coef, long T, int win, int hop, int nfft,
                                long wc, const float* hann, const float2* tw1, const float2* tw2, float* mag,
                                float* band, const int* lo, const int* hi, int n_bands, cudaStream_t st,
                                const ModVarlen* vl = nullptr);
// One clip of a ragged RMS-envelope launch (device descriptor, built on the host): the len samples at x + src, frames
// of frame_length samples every hop from -pad (samples outside [0, len) read as 0), T frames written from out + out.
// A work item is F consecutive frames of one clip; its span (F - 1) * hop + frame_length is staged in shared memory
// when it fits kRmsSpan floats, read from global memory otherwise.
struct RmsClip {
  long src, len, out, T;
  int frame_length, hop, pad, F;
};
constexpr int kRmsWarps = 8;      // one frame per warp at a time
constexpr int kRmsSpan = 12288;   // floats of a work item's staged span (48 KB)
// frames per work item of a clip (see RmsClip)
inline int rms_frames_per_item(int frame_length, int hop) {
  if (frame_length > kRmsSpan) return kRmsWarps;
  const int fit = (kRmsSpan - frame_length) / hop + 1, F = fit < 64 ? fit : 64;
  return F >= kRmsWarps ? F - F % kRmsWarps : F;
}
// Clip c owns work items [first_item[c], first_item[c + 1]) (ceil(T / F) each).  x is float32 or (pcm16) int16 scaled
// by 1/32768 as pcm16_to_f32_kernel scales it.
cudaError_t rms_varlen_launch(const void* x, int pcm16, const RmsClip* clips, const unsigned* first_item, long n_clips,
                              long n_items, float* out, cudaStream_t st);
cudaError_t fill_i32_launch(int* p, long n, int v, cudaStream_t st);
cudaError_t hilbert_envelope_launch(const float* x, long n_clips, long n, long stride, float* amp, long amp_stride,
                                    int sm_count, cudaStream_t st);
bool hilbert_fft_supported(long n);
cudaError_t hilbert_fft_launch(const float* x, long n_clips, long n, long stride, float* amp, long amp_stride,
                               cudaStream_t st);
cudaError_t find_peaks_launch(const double* x, long rows, long T, long stride, int minima, int max_peaks, int* idx,
                              int* count, cudaStream_t st);
cudaError_t pcm16_to_f32_launch(const int16_t* x, long n, float* y, cudaStream_t st);
// One clip of a ragged resampling launch (device descriptor, built on the host).  Output sample m of the clip is
// y_full[m + n_pre_remove] of upfirdn(h, x, up, down) over the clip's n_in samples at x + src; a plan-rate clip
// (copy != 0) is copied instead.  The clip's filter is h[tap0 .. tap0 + len_h) of the launch's tap table.
struct RsClip {
  long src, n_in, n_pre_remove, n_out, tap0;
  int up, down, len_h, copy;
};
constexpr int kRsOut = 256;  // outputs per work item of resample_rows_launch (one per thread)
// Clip c owns work items [first_item[c], first_item[c + 1]) (ceil(n_out / kRsOut) each); item k of the clip writes
// outputs [k * kRsOut, (k + 1) * kRsOut) of row c of y.  x is float32 or (pcm16) int16 scaled by 1/32768.
cudaError_t resample_rows_launch(const void* x, int pcm16, const RsClip* clips, const unsigned* first_item,
                                 long n_clips, long n_items, const float* h, float* y, long y_stride,
                                 cudaStream_t st);
// padded output rows -> packed blocks of the host-buffer bundle (see post_kernels.cu)
cudaError_t compact_rows_launch(const void* src, void* dst, int elem_bytes, long n_clips, int rows, int unit,
                                long pitch, const int* cnt, const long* off, cudaStream_t st);

// ---- host tables (host_tables.cpp)
struct MelSparse {
  std::vector<int> seg_start;  // n_mels + 2
  std::vector<float> w2;       // 2*F (falling, rising)
};
void host_window(int win_length, int n_fft, std::vector<float>& w);
void host_mel_dense(double sr, int n_fft, int n_mels, double fmin, double fmax, std::vector<float>& mel,
                    std::vector<double>& mel_f);
bool host_mel_sparse(const std::vector<float>& mel, const std::vector<double>& mel_f, double sr, int n_fft, int n_mels,
                     MelSparse& out);
struct MelGroups {
  std::vector<int> segtab;  // (first 4-bin group, first weight group) per segment, n_mels + 2 entries
  std::vector<int> segstep; // (groups of the segment, groups to step back before it) per segment, n_mels + 3 entries
  std::vector<float> w;     // 8 floats per weight group: 4 falling, 4 rising
  int n_groups = 0;
};
void host_mel_groups(const MelSparse& sp, int F, int n_mels, MelGroups& out);
void host_dct(int n_mfcc, int n_mels, std::vector<float>& d);
void host_twiddles(int n_fft, const StftGeometry& g, std::vector<float2>& tw1, std::vector<float2>& tw2);
int host_sos_zi(const double* sos, int n_sections, double* zi, int* padlen);

// opt a kernel into large dynamic shared memory once per device instead of on every launch
#define MMF_SMEM_ONCE(kfn, bytes)                                                                        \
  do {                                                                                                   \
    static bool done__[64] = {};                                                                         \
    int dev__ = 0;                                                                                       \
    cudaGetDevice(&dev__);                                                                               \
    if (dev__ < 0 || dev__ >= 64 || !done__[dev__]) {                                                    \
      cudaError_t e__ = cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (bytes)); \
      if (e__ != cudaSuccess) return e__;                                                                \
      if (dev__ >= 0 && dev__ < 64) done__[dev__] = true;                                                \
    }                                                                                                    \
  } while (0)

void set_error(const std::string& msg);
void count_launch(int n = 1);

}  // namespace mmf

struct mmf_plan {
  mmf_config cfg;
  int F;
  int sm_count;
  // tile geometry
  int TF, ppitch, pt_bufs, span_bufs, ctas_per_sm, lead, packed, mel_mma, threads = 256;
  size_t smem;
  // owners of every device table (d_*): upload() in c_api.cu allocates each one and records it here, the
  // trajectory-FFT tables (d_mod_*) in `mod_tables` because they are rebuilt; mmf_plan_destroy frees both
  std::vector<void*> tables, mod_tables;
  // generic n_fft: FP32 matrix-product DFT instead of the register FFT
  int generic = 0;
  float* d_dft_tab = nullptr;
  int dft_ld = 0;
  // device constants
  float* d_window = nullptr;
  float2* d_tw1 = nullptr;
  float2* d_tw2 = nullptr;
  int* d_seg = nullptr;
  int* d_band_split = nullptr;
  float2* d_mma_bw = nullptr;
  int* d_mma_pk8 = nullptr;
  int* d_mma_npair = nullptr;
  int* d_mma_tile = nullptr;
  int mma_n_tiles = 0;
  int* d_mma_units = nullptr;
  int mma_n_pairs = 0;
  size_t mel_tab_bytes = 0;
  float2* d_w2 = nullptr;
  int mel_groups = 0, mg_n = 0;  // grouped mel walk (bin-pair power tile)
  int2* d_mg_seg = nullptr;
  int2* d_mg_step = nullptr;
  float4* d_mg_w = nullptr;
  int win_lo = 0, win_hi = 16;  // 32-sample groups of the zero-padded window (n_fft = 512) that are not all zero
  int mel_tc_act = 0;        // non-empty mel bands (the rows of d_mel_tc)
  void* d_mel_tc = nullptr;  // bf16 [w1 ; w2] operand of the tcgen05 mel projection (null: not in use)
  float* d_dct = nullptr;  // [n_mels][nc_pad]
  float4* d_dct_bfrag = nullptr;  // DCT B fragments of the tensor-core MFCC kernel
  int nc_pad = 0;
  PFN_cuTensorMapEncodeTiled_v12000 encode = nullptr;
  void* d_dct_tc = nullptr;     // fp16 [Bhi ; Blo] operand of the tensor-core MFCC kernel
  int dct_tc_kp = 0;
  void* d_tc_btab = nullptr;    // fp16 DFT operand tables of the tensor-core transform (MMF_FLAG_TC_FFT)
  float2* d_tc_tw = nullptr;
  // tables of the trajectory FFT, rebuilt when (win, nfft, bands) change
  int mod_win = 0, mod_nfft = 0, mod_n_bands = -1;
  int mod_lo[16] = {0}, mod_hi[16] = {0};
  float* d_mod_hann = nullptr;
  float2* d_mod_tw1 = nullptr;
  float2* d_mod_tw2 = nullptr;
  int* d_mod_lo = nullptr;
  int* d_mod_hi = nullptr;
  void* d_mod_g = nullptr;  // fp16 [Ghi | Glo] operand of the tensor-core modulation spectrum
  int mod_g_kp = 0;
  // grow-only workspace for the composite entry points
  void* ws = nullptr;
  size_t ws_bytes = 0;
  void* host_ws = nullptr;  // workspace of the host-buffer entry points (they run on `streams`)
  size_t host_ws_bytes = 0;
  cudaStream_t streams[2] = {nullptr, nullptr};
};
