/*
 * mmf.h -- C ABI of the B200-native MFCC / cepstral-modulation hot path.
 *
 * The reference (aaron-randreth/modulation-mfcc) is pure Python and has no FFI;
 * each entry point below names the reference interface whose arithmetic it
 * replaces (paths relative to the reference checkout).  The Python drop-in
 * modules script/mfcc.py and script/calc.py bind these symbols with ctypes
 * (see INTEGRATION.md).
 *
 * Conventions
 *  - every function returns 0 on success or a negative mmf_status; the message
 *    is available from mmf_last_error() (thread-local);
 *  - pointers named *_dev are device pointers on the plan's device, *_host are
 *    host pointers; all buffers are caller-allocated, row-major, time innermost
 *    (librosa's [feature, T] layout per clip);
 *  - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *    device entry points are asynchronous on that stream;
 *  - there is no CPU fallback: without a CUDA device every compute entry point
 *    fails with MMF_ERR_CUDA.
 */
#ifndef MMF_H_
#define MMF_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MMF_VERSION 100

typedef enum {
  MMF_OK = 0,
  MMF_ERR_INVALID = -1,     /* bad argument (message says which) */
  MMF_ERR_UNSUPPORTED = -2, /* configuration outside the kernels' envelope */
  MMF_ERR_CUDA = -3,        /* CUDA runtime / driver error */
  MMF_ERR_TOO_SHORT = -4,   /* input shorter than the filter's padlen (scipy raises ValueError) */
  MMF_ERR_NOMEM = -5
} mmf_status;

/* Frame/spectrum configuration.  Mirrors the arguments librosa.feature.mfcc
 * receives at script/mfcc.py:387 plus the ones librosa defaults (n_mels = 128,
 * amin = 1e-10, top_db = 80). */
typedef struct {
  double sample_rate; /* sigSr */
  int32_t n_fft;      /* power of two in [256, 4096] */
  int32_t win_length; /* int(winLen * sigSr), <= n_fft            (script/mfcc.py:382) */
  int32_t hop_length; /* int(tStep * sigSr)                        (script/mfcc.py:384) */
  int32_t n_mels;     /* librosa default 128 when the reference is silent */
  int32_t n_mfcc;
  double fmin;        /* minFreq */
  double fmax;        /* maxFreq; may exceed Nyquist (script/main.py:739) */
  float amin;         /* 1e-10 */
  float top_db;       /* 80; negative disables the clamp */
  float preemph;      /* 0 = off (the reference applies none) */
  int32_t device;     /* CUDA device ordinal */
  int32_t flags;      /* MMF_FLAG_* */
} mmf_config;

#define MMF_FLAG_NO_TMA 1      /* load PCM spans with plain coalesced loads instead of TMA */
#define MMF_FLAG_SPLIT_SMEM 2  /* n_fft = 512: pair bins through shared memory instead of shuffles */
#define MMF_FLAG_SCALAR_FFT 8     /* one frame per thread group (scalar FP32) instead of two on packed FFMA2/FADD2 */
#define MMF_FLAG_MMA_MEL 16       /* mel projection on the tensor cores (mma.sync TF32 x3) instead of the sparse FP32 walk */
#define MMF_FLAG_MMA_DCT 32       /* clamp + DCT-II on the tensor cores (mma.sync TF32 x3) instead of scalar FP32 FMAs */
#define MMF_FLAG_UNFUSED_CHANGE 4 /* composite calls: separate filter / derivative kernels instead of the fused one */
#define MMF_FLAG_SEPARATE_MFCC 64 /* composite calls: clamp + DCT-II always as its own kernel */
#define MMF_FLAG_TC_FFT 256       /* n_fft = 512: the transform as tcgen05.mma kind::f16 GEMMs (fp16 x3 operand split,
                                     accumulators in tensor memory); mmf_stft_power only so far */
#define MMF_FLAG_NO_TC_MODSPEC 512 /* modulation spectrum always with the FP32 register FFT (default for win <= 128,
                                     nfft = 128: a tcgen05.mma kind::f16 GEMM with TMEM accumulators) */
#define MMF_FLAG_TC_DCT 1024       /* clamp + DCT-II (+ delta) as a tcgen05.mma kind::f16 GEMM over 128-frame tiles
                                     (n_mfcc <= 16, n_mels <= 96) instead of the FP32 FMA kernel; measured equal */
#define MMF_FLAG_MEL_WALK 2048     /* mel projection with the per-bin sparse walk on the [bin][frame] power tile instead of
                                      the grouped walk (four bins per step, packed FFMA2) on the bin-pair tile */
#define MMF_FLAG_NO_TC_MEL 4096    /* n_fft = 512, <= 112 non-empty bands: keep the mel projection on the CUDA cores (grouped walk)
                                      instead of the tcgen05.mma kind::f16 GEMM over 128-frame blocks (bf16 operand pairs,
                                      accumulators in tensor memory) */
#define MMF_FLAG_FOLD_MFCC 128    /* composite calls: clamp + DCT-II inside the per-clip kernel even when delta is wanted
                                     (default: folded only when no delta output is requested; measured in DESIGN.md) */

typedef struct mmf_plan mmf_plan;

int mmf_version(void);
const char* mmf_last_error(void);

/* Number of STFT frames librosa produces with center=True: 1 + n_samples / hop. */
int64_t mmf_num_frames(int64_t n_samples, int32_t n_fft, int32_t hop_length);

/* Host-only: the constant tables a plan uploads (no CUDA needed).  Any output
 * may be NULL.  window[n_fft] = periodic Hann(win_length) centred in n_fft;
 * mel[n_mels * (n_fft/2+1)] = librosa.filters.mel(htk=False, norm='slaney');
 * dct[n_mfcc * n_mels] = orthonormal DCT-II rows (scipy.fftpack.dct norm='ortho'). */
int mmf_host_tables(const mmf_config* cfg, float* window, float* mel, float* dct);

/* Host-only: scipy.signal.sosfilt_zi and sosfiltfilt's default padlen for a
 * cascade of n_sections biquads (sos row = b0 b1 b2 a0 a1 a2).  zi[n_sections*2]. */
int mmf_sos_zi(const double* sos, int32_t n_sections, double* zi, int32_t* padlen);

int mmf_plan_create(mmf_plan** out, const mmf_config* cfg);
int mmf_plan_destroy(mmf_plan* plan);

/* K1 alone: power spectrum |STFT|^2, [n_clips, n_fft/2+1, T] float32.
 * Replaces librosa.stft + abs**2 under script/mfcc.py:387. */
int mmf_stft_power(mmf_plan* plan, const float* pcm_dev, int64_t n_clips, int64_t n_samples, int64_t clip_stride,
                   float* power_dev, void* stream);

/* K1+K2 fused: log-mel spectrogram before the top_db clamp, [n_clips, n_mels, T]
 * float32, plus clipmax_dev[n_clips] (int32 keys of the per-clip maximum, consumed
 * by mmf_mfcc).  Replaces stft/abs**2/filters.mel/einsum/10*log10 under
 * script/mfcc.py:387. */
int mmf_logmel(mmf_plan* plan, const float* pcm_dev, int64_t n_clips, int64_t n_samples, int64_t clip_stride,
               float* logmel_dev, int32_t* clipmax_dev, void* stream);

/* K3: top_db clamp (in place on logmel_dev when clamp_in_place != 0) + DCT-II
 * -> mfcc_dev [n_clips, n_mfcc, T] float32; optional delta_dev (np.gradient along
 * time, unit spacing == calc.get_velocity(x, sr=1.0) at script/calc.py:642-645).
 * Replaces power_to_db's clamp and scipy.fftpack.dct under script/mfcc.py:387. */
int mmf_mfcc(mmf_plan* plan, float* logmel_dev, const int32_t* clipmax_dev, int64_t n_clips, int64_t T,
             float* mfcc_dev, float* delta_dev, int32_t clamp_in_place, void* stream);

/* K4: scipy.signal.sosfiltfilt(sos, x) along time for `rows` rows
 * (script/mfcc.py:402, :421, :111).  x is float32 or float64; y is float64.
 * Row r starts at x + r*x_row_stride (elements). */
int mmf_sosfiltfilt(mmf_plan* plan, const void* x_dev, int32_t x_is_f32, int64_t rows, int64_t T,
                    int64_t x_row_stride, const double* sos_host, int32_t n_sections, double* y_dev,
                    int64_t y_row_stride, void* stream);

/* K5: derivative along time of `rows_per_clip` float64 rows then
 * sqrt(sum_rows d^2) / rows_per_clip -> tot_dev[n_clips, T] float64
 * (script/mfcc.py:405-415).  method 0 = np.gradient, 1 = savgol(3, 2, deriv=1, 'interp'). */
int mmf_delta_norm(mmf_plan* plan, const double* x_dev, int64_t n_clips, int32_t rows_per_clip, int64_t T,
                   int32_t method, double* tot_dev, void* stream);

/* Generic zero-phase FIR: scipy.signal.filtfilt(b, 1, x) (script/mfcc.py:126). */
int mmf_fir_filtfilt(mmf_plan* plan, const double* x_dev, int64_t rows, int64_t T, const double* b_host,
                     int32_t n_taps, double* y_dev, double* work_dev /* rows*(T+6*n_taps) */, void* stream);

/* Generic banded stencil with dense boundary rows: interior
 * y[t] = sum_o c[o+half]*x[t+o]; the first/last n_edge outputs are
 * edge_l/edge_r [n_edge, n_edge_in] applied to the first/last n_edge_in inputs.
 * Covers np.gradient, savgol_filter(mode='interp') and findiff stencils
 * (script/calc.py:635-645, script/mfcc.py:130,411). */
int mmf_stencil(mmf_plan* plan, const double* x_dev, int64_t rows, int64_t T, const double* coef_host, int32_t half,
                const double* edge_l_host, const double* edge_r_host, int32_t n_edge, int32_t n_edge_in,
                double* y_dev, void* stream);

/* K6: modulation spectrum of MFCC trajectories (extension, SURVEY.md Appendix B):
 * windows of win frames every hop frames, mean removed, periodic Hann, zero padded
 * to nfft (power of two <= 4096), magnitude of the real FFT ->
 * mag_dev [n_clips, n_coef, n_win, nfft/2+1]; band energies summed over
 * coefficients -> band_dev [n_clips, n_win, n_bands] for bins
 * [band_lo[b], band_hi[b]).  Either output may be NULL. */
int mmf_modspec(mmf_plan* plan, const float* mfcc_dev, int64_t n_clips, int32_t n_coef, int64_t T, int32_t win,
                int32_t hop, int32_t nfft, float* mag_dev, float* band_dev, const int32_t* band_lo_host,
                const int32_t* band_hi_host, int32_t n_bands, void* stream);

/* mmf_modspec for clips of different lengths in one call.  Clip i is n_coef rows of T_host[i] valid frames at
 * mfcc_dev + i * n_coef * pitch, rows pitch frames apart (0 <= T_host[i] <= pitch); frames >= T_host[i] are never
 * read into any output.  n_win_i = 1 + (T_host[i] - win) / hop (0 when T_host[i] < win), W = max n_win_i; outputs
 * are padded to W: optional mag_dev [n_clips, n_coef, W, nfft/2+1] and band_dev [n_clips, W, n_bands].  Windows
 * [0, n_win_i) of clip i are bit-identical to mmf_modspec on that clip alone (n_clips = 1, T = T_host[i], rows
 * contiguous); every element at a window >= n_win_i is 0.  W = 0 launches nothing.  All arguments are checked
 * before anything is launched (the lengths and the geometry without a plan or a device: a bad T_host[i] fails
 * with MMF_ERR_INVALID, the message naming its index).  Each clip takes the kernel its own call takes; clips on
 * the tcgen05 and the clip-resident kernels run in one launch per kernel for the whole batch (more than 2^31 - 1
 * work items: MMF_ERR_UNSUPPORTED), the others one by one. */
int mmf_modspec_varlen(mmf_plan* plan, const float* mfcc_dev, int64_t n_clips, int32_t n_coef, const int64_t* T_host,
                       int64_t pitch, int32_t win, int32_t hop, int32_t nfft, float* mag_dev, float* band_dev,
                       const int32_t* band_lo_host, const int32_t* band_hi_host, int32_t n_bands, void* stream);

/* RMS envelope: librosa.feature.rms(frame_length, hop_length, center,
 * pad_mode='constant') (script/calc.py:326-331, script/mfcc.py:247) ->
 * rms_dev [n_clips, T_rms] float32, T_rms = 1 + (n + 2*pad - frame_length)/hop.
 * Each frame is summed in one fixed order (lane l of a warp: fmaf over samples l, l + 32, ...; then an xor-shuffle
 * tree 16, 8, 4, 2, 1; then sqrtf(s / frame_length)), so a row's bits do not depend on its batch. */
int mmf_rms(mmf_plan* plan, const float* pcm_dev, int64_t n_clips, int64_t n_samples, int64_t clip_stride,
            int32_t frame_length, int32_t hop_length, int32_t center, float* rms_dev, void* stream);

/* Host-only: output offsets of the RMS envelopes of a packed batch (no plan, no device).  Clip i is samples
 * [offsets_host[i], offsets_host[i+1]) with geom_host[2i] = frame_length_i, geom_host[2i+1] = hop_i (in samples at the
 * clip's own rate); pad_i = center ? frame_length_i / 2 : 0 and T_amp_i = 1 + (len_i + 2 pad_i - frame_length_i) /
 * hop_i.  amp_off_host[n_clips+1] = prefix sums of T_amp_i.  The offsets are checked as mmf_features_host_varlen
 * checks them; frame_length or hop < 1 fails with MMF_ERR_INVALID, a clip shorter than its frame without center with
 * MMF_ERR_TOO_SHORT, the message naming the clip. */
int mmf_amp_varlen_sizes(int64_t n_clips, const int64_t* offsets_host, const int32_t* geom_host, int32_t center,
                         int64_t* amp_off_host);

/* mmf_rms for packed clips of different lengths and frame geometries, in one launch: clip i of the packed float32
 * x_dev[offsets_host[i] .. offsets_host[i+1]) with geom_host[2i .. 2i+1] goes to amp_dev[amp_off[i] .. amp_off[i+1])
 * (mmf_amp_varlen_sizes).  Each block is bit-identical to mmf_rms on that clip alone.  The checks are those of
 * mmf_amp_varlen_sizes, before anything is launched.  Asynchronous on `stream` (the descriptors are copied from
 * pageable memory before it returns). */
int mmf_rms_varlen(mmf_plan* plan, const float* x_dev, int64_t n_clips, const int64_t* offsets_host,
                   const int32_t* geom_host, int32_t center, float* amp_dev, void* stream);

/* Parameters of the post-MFCC part of get_MFCCS_change (script/mfcc.py:393-425). */
typedef struct {
  int32_t remove_first; /* removeFirst */
  int32_t diff_method;  /* 0 = 'grad', 1 = Savitzky-Golay */
  int32_t n_sections;   /* Butterworth low-pass of the MFCC rows (script/mfcc.py:398-402) */
  double sos[16 * 6];
  int32_t out_kind;     /* 0 = sosfiltfilt with out_sos (outFilter None or 'iir'), 1 = none (raw change) */
  int32_t out_n_sections;
  double out_sos[16 * 6];
} mmf_change_params;

/* Whole get_MFCCS_change for a batch resident on the device: PCM -> totChange
 * [n_clips, T] float64.  Optional outputs (NULL to skip): logmel_dev (clamped),
 * mfcc_dev, delta_dev.  Intermediate buffers come from the plan's workspace. */
int mmf_mfcc_change(mmf_plan* plan, const float* pcm_dev, int64_t n_clips, int64_t n_samples, int64_t clip_stride,
                    const mmf_change_params* prm, double* tot_dev, float* logmel_dev, float* mfcc_dev,
                    float* delta_dev, void* stream);

/* mmf_mfcc_change for clips of different lengths in one call.  Clip i is the n_samples_host[i] samples at
 * pcm_dev + i * clip_stride (1 <= n_samples_host[i] <= clip_stride); samples past a clip's length are never
 * read as anything but zero, whatever the buffer holds there.  T_i = mmf_num_frames(n_samples_host[i], ...),
 * T_max = max T_i; outputs are padded to T_max: tot_dev [n_clips, T_max], optional logmel_dev / mfcc_dev /
 * delta_dev [n_clips, n_mels | n_mfcc, T_max].  Frames [0, T_i) of clip i are bit-identical to
 * mmf_mfcc_change on that clip alone (n_clips = 1, n_samples = n_samples_host[i]); every element at a frame
 * >= T_i is 0.  A clip with T_i <= padlen fails with MMF_ERR_TOO_SHORT, the message naming its index; all
 * arguments are checked before anything is launched.  Clips on the default kernel routes run in one launch
 * per stage for the whole batch; the others (generic n_fft, the non-default MFCC / change flags, rows longer
 * than the fused kernel takes) run one by one. */
int mmf_mfcc_change_varlen(mmf_plan* plan, const float* pcm_dev, int64_t n_clips, const int64_t* n_samples_host,
                           int64_t clip_stride, const mmf_change_params* prm, double* tot_dev, float* logmel_dev,
                           float* mfcc_dev, float* delta_dev, void* stream);

/* Second half of mmf_mfcc_change, for callers that already hold the log-mel
 * (mmf_logmel): clamp -> MFCC (+delta) -> zero-phase Butterworth -> derivative +
 * norm -> output filter (script/mfcc.py:387 tail .. :425). */
int mmf_change_from_logmel(mmf_plan* plan, float* logmel_dev, const int32_t* clipmax_dev, int64_t n_clips, int64_t T,
                           const mmf_change_params* prm, double* tot_dev, float* mfcc_dev, float* delta_dev,
                           int32_t clamp_in_place, void* stream);

/* Modulation-spectrum parameters for the host-buffer bundle call (win = 0: none). */
typedef struct {
  int32_t win, hop, nfft;
  int32_t n_bands;
  int32_t band_lo[16];
  int32_t band_hi[16];
} mmf_modspec_params;

/* The whole feature bundle with HOST buffers in and out: PCM is copied
 * host->device in chunks overlapped with compute on two streams, every requested
 * output is copied back, and the call returns after synchronising.  tot_host is
 * required; mfcc_host / delta_host [n_clips, n_mfcc, T], mag_host
 * [n_clips, n_mfcc, n_win, nfft/2+1] and band_host [n_clips, n_win, n_bands] are
 * optional (NULL).  Pinned host memory makes the copies truly asynchronous. */
int mmf_features_host(mmf_plan* plan, const float* pcm_host, int64_t n_clips, int64_t n_samples, int64_t clip_stride,
                      const mmf_change_params* prm, const mmf_modspec_params* mod, double* tot_host, float* mfcc_host,
                      float* delta_host, float* mag_host, float* band_host);

/* mmf_features_host for 16-bit PCM as it sits in a WAV file: the int16 samples cross PCIe as they are
 * (half the bytes) and are scaled to float32 = x / 32768 on the device, exactly what
 * librosa.load / soundfile does on the CPU before the path starts (script/mfcc.py:373). */
int mmf_features_host_pcm16(mmf_plan* plan, const int16_t* pcm16_host, int64_t n_clips, int64_t n_samples,
                            int64_t clip_stride, const mmf_change_params* prm, const mmf_modspec_params* mod,
                            double* tot_host, float* mfcc_host, float* delta_host, float* mag_host,
                            float* band_host);

/* Host-only: output offsets of a packed batch (no plan, no device).  Clip i is samples
 * [offsets_host[i], offsets_host[i+1]) of the packed input.  frame_off[n_clips+1] = prefix sums of T_i =
 * mmf_num_frames(len_i, ...); win_off[n_clips+1] = prefix sums of n_win_i (all 0 when mod is NULL or win = 0).
 * The offsets are checked as mmf_features_host_varlen checks them. */
int mmf_features_varlen_sizes(const mmf_config* cfg, const mmf_modspec_params* mod, int64_t n_clips,
                              const int64_t* offsets_host, int64_t* frame_off_host, int64_t* win_off_host);

/* mmf_features_host for clips of different lengths packed back to back in one host buffer.
 *  - Input: clip i is pcm_host[offsets_host[i] .. offsets_host[i+1]).  Offsets are non-decreasing from
 *    offsets_host[0] >= 0 and every clip has at least 1 sample.  Nothing before offsets_host[0] or after
 *    offsets_host[n_clips] is read, and no sample of one clip reaches another clip's outputs.
 *  - Outputs are packed in clip order, with no padding.  With F_i = frame_off[i], W_i = win_off[i]
 *    (mmf_features_varlen_sizes): tot_host[F_i .. F_i + T_i); mfcc_host / delta_host: clip i's [n_mfcc, T_i] block
 *    at n_mfcc * F_i; mag_host: its [n_mfcc, n_win_i, nfft/2+1] block at n_mfcc * (nfft/2+1) * W_i; band_host: its
 *    [n_win_i, n_bands] block at n_bands * W_i.  Optional outputs and their NULL rules are those of
 *    mmf_features_host.
 *  - Each clip's blocks are bit-identical to mmf_features_host (or _pcm16) on that clip alone, whatever chunk the
 *    clip lands in and whoever its neighbours are.  For clips of equal length the packed layout is the padded one,
 *    and the results equal mmf_features_host on the [n_clips, N] array byte for byte.
 *  - Everything is checked before anything is queued: the offsets first, without a plan or a device (NULL or
 *    decreasing offsets and empty clips fail with MMF_ERR_INVALID, the message naming the clip); a clip too short
 *    for the filters fails with MMF_ERR_TOO_SHORT, naming its index.
 *  - The batch runs in chunks of consecutive clips over the plan's two streams (copy in, compute and copy out
 *    overlap); the call returns after draining both, on every exit. */
int mmf_features_host_varlen(mmf_plan* plan, const float* pcm_host, int64_t n_clips, const int64_t* offsets_host,
                             const mmf_change_params* prm, const mmf_modspec_params* mod, double* tot_host,
                             float* mfcc_host, float* delta_host, float* mag_host, float* band_host);
/* The same for 16-bit PCM, scaled to float32 = x / 32768 on the device as mmf_features_host_pcm16 does. */
int mmf_features_host_varlen_pcm16(mmf_plan* plan, const int16_t* pcm16_host, int64_t n_clips,
                                   const int64_t* offsets_host, const mmf_change_params* prm,
                                   const mmf_modspec_params* mod, double* tot_host, float* mfcc_host,
                                   float* delta_host, float* mag_host, float* band_host);

/* How one clip of a packed batch reaches the plan's rate.  up = down = 1: the clip is already at the plan's rate and is
 * taken as it is (n_out = its length; tap0, len_h and n_pre_remove are not read).  Otherwise the clip is resampled
 * exactly as mmf_resample_poly resamples a row with the filter h[tap0 .. tap0 + len_h) of the call's tap table
 * (design: plan.design_resample_filter), n_pre_remove and n_out = ceil(len * up / down). */
typedef struct {
  int32_t up, down;
  int64_t tap0;
  int32_t len_h;
  int64_t n_pre_remove, n_out;
} mmf_resample_clip;

/* mmf_features_host_varlen for packed clips that each arrive at their own sample rate.
 *  - Input: clip i is pcm_host[offsets_host[i] .. offsets_host[i+1]), float32 or (pcm16 != 0) int16 scaled by
 *    1/32768; rs_host[i] says how it reaches the plan's rate, with taps from h_host[n_h] (NULL when every clip is at
 *    the plan's rate).  Each clip's native samples cross PCIe once and are resampled on the device straight into the
 *    rows the ragged path reads, in one staging launch per chunk whatever its mix of rates.
 *  - Outputs are packed as mmf_features_host_varlen packs them, with T_i = mmf_num_frames(n_out_i, ...): frame and
 *    window offsets come from mmf_features_varlen_sizes given the prefix sums of n_out_i as offsets.
 *  - Each clip's blocks are bit-identical to mmf_features_host on mmf_resample_poly's output for that clip alone
 *    (after mmf_pcm16_to_f32 for int16), whatever chunk the clip lands in and whoever its neighbours are; a plan-rate
 *    clip's blocks equal mmf_features_host_varlen's.
 *  - Everything is checked before anything is queued, the offsets and descriptors without a plan or a device (the
 *    message names the clip): the offsets as mmf_features_host_varlen checks them, up, down >= 1, n_out =
 *    ceil(len * up / down) (= len at the plan's rate), and for a resampled clip 1 <= len_h <= 2^22, tap0 >= 0,
 *    tap0 + len_h <= n_h and n_pre_remove >= 0 (MMF_ERR_INVALID).  A clip too short for the filters after resampling
 *    fails with MMF_ERR_TOO_SHORT, naming its index. */
int mmf_features_host_varlen_resampled(mmf_plan* plan, const void* pcm_host, int32_t pcm16, int64_t n_clips,
                                       const int64_t* offsets_host, const mmf_resample_clip* rs_host,
                                       const float* h_host, int64_t n_h, const mmf_change_params* prm,
                                       const mmf_modspec_params* mod, double* tot_host, float* mfcc_host,
                                       float* delta_host, float* mag_host, float* band_host);

/* The resampling stage of mmf_features_host_varlen_resampled alone, on the device: clip i of the packed float32
 * x_dev[offsets_host[i] .. offsets_host[i+1]) goes to y_dev + i * y_stride (rs_host[i].n_out samples; the rest of the
 * row is not written; y_stride >= max n_out).  The checks are those of mmf_features_host_varlen_resampled.  One
 * launch, asynchronous on `stream` (the call's descriptors and taps are copied from pageable memory before it
 * returns). */
int mmf_resample_varlen(mmf_plan* plan, const float* x_dev, int64_t n_clips, const int64_t* offsets_host,
                        const mmf_resample_clip* rs_host, const float* h_host, int64_t n_h, float* y_dev,
                        int64_t y_stride, void* stream);

/* The RMS amplitude envelope in the host-buffer bundle (calculate_amplitude_envelope, script/calc.py:221-343, method
 * 'RMS', outFilter None or 'iir').  out_n_sections = 0: the raw envelope only; otherwise out_sos holds the
 * zero-phase output filter (designed at 1 / hopLen, as applyFilter designs it). */
typedef struct {
  int32_t center;
  int32_t out_n_sections;
  double out_sos[16 * 6];
} mmf_amp_params;

/* mmf_features_host_varlen_resampled plus each clip's RMS envelope at its native rate.
 *  - rs_host and h_host may be NULL: every clip is then at the plan's rate, as in mmf_features_host_varlen(_pcm16).
 *  - amp = NULL: exactly mmf_features_host_varlen_resampled (amp_host and amp_filt_host must then be NULL).
 *  - Otherwise the envelope of clip i is taken from its native samples (float32, or int16 scaled by 1/32768) with
 *    geom_host[2i] = frame_length_i, geom_host[2i+1] = hop_i and amp->center; amp_host (float32) and amp_filt_host
 *    (float64, the envelope through amp->out_sos; needs out_n_sections > 0) receive it packed at amp_off
 *    (mmf_amp_varlen_sizes).  Either may be NULL.  Each clip's blocks are bit-identical to mmf_rms, then
 *    mmf_sosfiltfilt (x_is_f32 = 1) on that clip alone, whatever chunk it lands in.
 *  - The MFCC side and its checks are unchanged.  The amplitude checks are those of mmf_amp_varlen_sizes; with a
 *    filter, an envelope of at most padlen frames fails with MMF_ERR_TOO_SHORT naming the clip, before anything is
 *    queued.
 *  - Per chunk, the envelope is one launch reading the chunk's copied samples and, with a filter, one more for every
 *    envelope the chunk-parallel filter takes; longer envelopes are filtered one by one. */
int mmf_features_host_varlen_amp(mmf_plan* plan, const void* pcm_host, int32_t pcm16, int64_t n_clips,
                                 const int64_t* offsets_host, const mmf_resample_clip* rs_host, const float* h_host,
                                 int64_t n_h, const mmf_change_params* prm, const mmf_modspec_params* mod,
                                 const mmf_amp_params* amp, const int32_t* geom_host, double* tot_host,
                                 float* mfcc_host, float* delta_host, float* mag_host, float* band_host,
                                 float* amp_host, double* amp_filt_host);

/* Hilbert amplitude envelope |scipy.signal.hilbert(x)| of each row (script/calc.py:284-286, method 'Hilb'),
 * any length n <= 2^26 (an hour at 16 kHz): O(n log n) -- the length-n transforms scipy runs are evaluated as
 * Bluestein chirp transforms over a power-of-two FFT in float64, the rows as one batch of mmf_hilbert_varlen;
 * signals of at most 4096 samples use the equivalent direct circular convolution with the discrete Hilbert
 * kernel. */
int mmf_hilbert_envelope(mmf_plan* plan, const float* x_dev, int64_t n_clips, int64_t n, int64_t x_stride,
                         float* amp_dev, int64_t amp_stride, void* stream);

/* mmf_hilbert_envelope for packed clips of different lengths: clip i of the packed float32
 * x_dev[offsets_host[i] .. offsets_host[i+1]) has its envelope at the same range of amp_dev, counted from
 * offsets_host[0] (amp_dev holds offsets_host[n_clips] - offsets_host[0] floats).  Each block is bit-identical to
 * mmf_hilbert_envelope on that clip alone.  Clips of more than 4096 samples run together in a fixed number of
 * launches (the chirp tables once per distinct length, then five FFTs of two or three pass-group launches each),
 * in sub-batches of bounded scratch; shorter ones one by one.  The offsets are checked as mmf_rms_varlen checks
 * them; a clip over 2^26 samples fails with MMF_ERR_UNSUPPORTED naming the clip; every check runs before anything
 * is queued.  Asynchronous on `stream`. */
int mmf_hilbert_varlen(mmf_plan* plan, const float* x_dev, int64_t n_clips, const int64_t* offsets_host,
                       float* amp_dev, void* stream);

/* The envelope of the host-buffer bundle (calculate_amplitude_envelope, script/calc.py:221-343, outFilter None or
 * 'iir'): method MMF_ENV_RMS (frame geometry per clip, center) or MMF_ENV_HILBERT (one output per sample; center
 * and the geometry are not read).  out_n_sections and out_sos as in mmf_amp_params. */
#define MMF_ENV_RMS 0
#define MMF_ENV_HILBERT 1
typedef struct {
  int32_t method;
  int32_t center;
  int32_t out_n_sections;
  double out_sos[16 * 6];
} mmf_env_params;

/* Host-only: output offsets of the envelopes of a packed batch.  RMS: mmf_amp_varlen_sizes with env->center.
 * Hilbert: amp_off_host = prefix sums of the clip lengths (geom_host may be NULL); a clip over 2^26 samples fails
 * with MMF_ERR_UNSUPPORTED naming the clip.  An unknown method fails with MMF_ERR_INVALID. */
int mmf_env_varlen_sizes(int64_t n_clips, const int64_t* offsets_host, const mmf_env_params* env,
                         const int32_t* geom_host, int64_t* amp_off_host);

/* mmf_features_host_varlen_amp with the envelope method in env (mmf_features_host_varlen_amp is this call with
 * method MMF_ENV_RMS).  The Hilbert envelope of each chunk is taken from its copied native samples (float32, or
 * int16 scaled by 1/32768) on the chunk's stream: equal, bit for bit, to mmf_hilbert_envelope on the clip alone
 * and, with a filter, then to mmf_sosfiltfilt (x_is_f32 = 1) on that envelope; these long rows are filtered one by
 * one.  With a filter, an envelope of at most padlen samples fails with MMF_ERR_TOO_SHORT naming the clip, before
 * anything is queued. */
int mmf_features_host_varlen_env(mmf_plan* plan, const void* pcm_host, int32_t pcm16, int64_t n_clips,
                                 const int64_t* offsets_host, const mmf_resample_clip* rs_host, const float* h_host,
                                 int64_t n_h, const mmf_change_params* prm, const mmf_modspec_params* mod,
                                 const mmf_env_params* env, const int32_t* geom_host, double* tot_host,
                                 float* mfcc_host, float* delta_host, float* mag_host, float* band_host,
                                 float* amp_host, double* amp_filt_host);

/* The 'fir' and 'sg' output filters of applyFilter (script/mfcc.py:113-131), as coefficients designed on the host.
 * MMF_FILT_FIR: scipy.signal.filtfilt(taps, 1, x), n_taps in [1, 4096].  MMF_FILT_SG: a banded stencil with dense
 * edge rows, as mmf_stencil takes it (savgol_filter(mode='interp'), np.gradient, findiff).  All pointers are host
 * pointers; the fields the kind does not use are ignored. */
#define MMF_FILT_FIR 0
#define MMF_FILT_SG 1
typedef struct mmf_out_filter {
  int32_t kind;          /* MMF_FILT_FIR or MMF_FILT_SG */
  int32_t n_taps;        /* FIR */
  const double* taps;    /* FIR: b[n_taps] */
  int32_t half;          /* SG: y[t] = sum_o coef[o + half] * x[t + o] in the interior */
  const double* coef;    /* SG: [2 * half + 1] */
  int32_t n_edge;        /* SG: the first / last n_edge outputs are edge_l / edge_r ... */
  int32_t n_edge_in;     /* ... [n_edge, n_edge_in] applied to the first / last n_edge_in inputs; n_edge >= half */
  const double* edge_l;
  const double* edge_r;
} mmf_out_filter;

/* Host-only: the checks of mmf_filter_varlen for n_rows rows of T_host[i] samples, without a plan or a device.
 * FIR: T_i <= 3 * n_taps fails with MMF_ERR_TOO_SHORT and filtfilt's padlen message; SG: T_i < n_edge_in or
 * T_i < 2 * n_edge fails with MMF_ERR_TOO_SHORT.  Both name the row ("clip i: ").  A bad kind, tap count or edge
 * shape fails with MMF_ERR_INVALID or MMF_ERR_UNSUPPORTED. */
int mmf_filter_varlen_check(const mmf_out_filter* filt, int64_t n_rows, const int64_t* T_host);

/* The output filter filt over n_rows rows of any lengths, in a fixed number of launches (FIR: 2, SG: 1) whatever the
 * row count: row i is the T_host[i] samples at x_dev + x_off_host[i] (float64, or x_is_f32 float32), its T_host[i]
 * float64 outputs go to y_dev + y_off_host[i] (offsets in elements).  A padded [B, T_max] batch and a packed one
 * are the same call.  Each row's output equals, bit for bit, mmf_fir_filtfilt / mmf_stencil on that row alone.
 * Every check (mmf_filter_varlen_check) runs before anything is queued; the descriptors and coefficients are copied
 * before the call returns, which is asynchronous on `stream`.  FIR scratch comes from the stream-ordered pool. */
int mmf_filter_varlen(mmf_plan* plan, const mmf_out_filter* filt, const void* x_dev, int32_t x_is_f32, int64_t n_rows,
                      const int64_t* x_off_host, const int64_t* T_host, double* y_dev, const int64_t* y_off_host,
                      void* stream);

/* mmf_features_host_varlen_env with an output filter on the MFCC-change curve.  change_out NULL: exactly
 * mmf_features_host_varlen_env.  Otherwise prm->out_kind must be 1 (the raw curve; else MMF_ERR_INVALID): each
 * chunk's raw curves are filtered by change_out (mmf_filter_varlen over the chunk's padded rows) and tot_host
 * receives the filtered curves, each equal to mmf_filter_varlen on that clip's raw curve alone.  A clip too short
 * for the change stage's Butterworth filter reports that first; otherwise a curve too short for change_out fails
 * as mmf_filter_varlen_check fails, naming the clip, before anything is queued. */
int mmf_features_host_varlen_out(mmf_plan* plan, const void* pcm_host, int32_t pcm16, int64_t n_clips,
                                 const int64_t* offsets_host, const mmf_resample_clip* rs_host, const float* h_host,
                                 int64_t n_h, const mmf_change_params* prm, const mmf_modspec_params* mod,
                                 const mmf_env_params* env, const int32_t* geom_host,
                                 const mmf_out_filter* change_out, double* tot_host, float* mfcc_host,
                                 float* delta_host, float* mag_host, float* band_host, float* amp_host,
                                 double* amp_filt_host);

/* Local extrema of each float64 row with scipy.signal.find_peaks' default semantics (strictly higher
 * than both neighbours; a flat top reports its middle sample; end samples never qualify) -- the
 * landmark step the GUI runs on the curve (script/main.py:1566, :1601; script/calc.py:669, :681).
 * idx_dev [rows, max_peaks] receives the indices in ascending order, count_dev [rows] the number
 * found (may exceed max_peaks: only the first max_peaks are stored).  minima != 0: peaks of -x. */
int mmf_find_peaks(mmf_plan* plan, const double* x_dev, int64_t rows, int64_t T, int64_t row_stride, int32_t minima,
                   int32_t max_peaks, int32_t* idx_dev, int32_t* count_dev, void* stream);

/* Device-side PCM16 -> float32 in [-1, 1): y = x / 32768 (script/mfcc.py:373, :284 decode step). */
int mmf_pcm16_to_f32(mmf_plan* plan, const int16_t* pcm16_dev, int64_t n, float* pcm_dev, void* stream);

/* Rational-rate polyphase resampler with scipy.signal.resample_poly / upfirdn semantics, one launch for all rows
 * (n_clips rows of n_in samples, x_stride apart):
 * y_full[m] = sum_i h[m*down - i*up] * x[i];  y = y_full[n_pre_remove : n_pre_remove + n_out].
 * h (already scaled by `up` and zero-padded as resample_poly does) is designed on the host.  The
 * step before the path: librosa.load(path, sr=sigSr) at script/mfcc.py:373, :284 (librosa uses
 * soxr_hq there; this resampler is NOT bit-identical to it, see DESIGN.md). */
int mmf_resample_poly(mmf_plan* plan, const float* x_dev, int64_t n_clips, int64_t n_in, int64_t x_stride,
                      const float* h_host, int32_t len_h, int32_t up, int32_t down, int64_t n_pre_remove, int64_t n_out,
                      float* y_dev, int64_t y_stride, void* stream);

/* Same as mmf_features_host with only totChange (and optionally MFCC) returned:
 * HOST buffers in and out (the call the Python drop-in makes for a numpy
 * array): copies PCM host->device in chunks overlapped with compute, runs the
 * path, copies totChange (and mfcc_host if not NULL) back, synchronises. */
int mmf_mfcc_change_host(mmf_plan* plan, const float* pcm_host, int64_t n_clips, int64_t n_samples,
                         int64_t clip_stride, const mmf_change_params* prm, double* tot_host, float* mfcc_host);

/* sizeof() of the ABI structs as this library was compiled (0: mmf_config,
 * 1: mmf_change_params, 2: mmf_modspec_params, 3: mmf_resample_clip, 4: mmf_amp_params, 5: mmf_env_params,
 * 6: mmf_out_filter) so
 * bindings can verify their layout. */
int mmf_abi_sizeof(int32_t which);

/* Number of kernels this library has launched on the calling thread since the
 * last reset (bench.py reports it as gpu_launches). */
int64_t mmf_launch_count(int32_t reset);

#ifdef __cplusplus
}
#endif
#endif /* MMF_H_ */
