// extern "C" surface of libmmf_b200.so (declared in include/mmf.h).
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <cudaTypedefs.h>

#include "mmf_internal.h"
#include "sos_par.cuh"

namespace mmf {

static thread_local std::string g_err;
static thread_local long g_launches = 0;

void set_error(const std::string& msg) { g_err = msg; }
void count_launch(int n) { g_launches += n; }

static int fail(int code, const std::string& msg) {
  set_error(msg);
  return code;
}
static int cuda_fail(cudaError_t e, const char* where) {
  return fail(MMF_ERR_CUDA, std::string(where) + ": " + cudaGetErrorString(e));
}
// scipy's message; clip >= 0: a batch's, naming the clip
static int too_short(int padlen, int64_t clip = -1) {
  const std::string at = clip < 0 ? "" : "clip " + std::to_string(clip) + ": ";
  return fail(MMF_ERR_TOO_SHORT, at + "The length of the input vector x must be greater than padlen, which is " +
                                     std::to_string(padlen) + ".");
}
#define MMF_CUDA(call)                                   \
  do {                                                   \
    cudaError_t e__ = (call);                            \
    if (e__ != cudaSuccess) return cuda_fail(e__, #call); \
  } while (0)

static int validate_cfg(const mmf_config* c) {
  if (!c) return fail(MMF_ERR_INVALID, "config is NULL");
  if (c->n_fft < 16 || c->n_fft > 4096) return fail(MMF_ERR_UNSUPPORTED, "n_fft must be in [16, 4096]");
  if (c->win_length < 1 || c->win_length > c->n_fft)
    return fail(MMF_ERR_INVALID, "Target size (n_fft) must be at least input size (win_length)");
  if (c->hop_length < 1) return fail(MMF_ERR_INVALID, "hop_length must be a positive integer");
  if (c->n_mels < 1 || c->n_mels > 512) return fail(MMF_ERR_UNSUPPORTED, "n_mels must be in [1, 512]");
  if (c->n_mfcc < 1 || c->n_mfcc > 128 || c->n_mfcc > c->n_mels)
    return fail(MMF_ERR_UNSUPPORTED, "n_mfcc must be in [1, min(128, n_mels)]");
  if (!(c->sample_rate > 0)) return fail(MMF_ERR_INVALID, "sample_rate must be positive");
  if (!(c->fmax > c->fmin) || c->fmin < 0) return fail(MMF_ERR_INVALID, "need 0 <= fmin < fmax");
  return MMF_OK;
}

// the only allocator of plan tables: copies `src` to new device memory that `owner` (a list of the plan) frees.  A
// no-op once `e` holds an error, so that a run of uploads is checked once at its end.
template <typename D, typename T>
static void upload(cudaError_t& e, std::vector<void*>& owner, D** dst, const std::vector<T>& src) {
  void* d = nullptr;
  if (e != cudaSuccess || (e = cudaMalloc(&d, std::max<size_t>(1, src.size()) * sizeof(T))) != cudaSuccess) return;
  owner.push_back(d);
  *dst = static_cast<D*>(d);
  e = cudaMemcpy(d, src.data(), src.size() * sizeof(T), cudaMemcpyHostToDevice);
}

static int ensure_ws(mmf_plan* p, size_t bytes) {
  if (bytes <= p->ws_bytes) return MMF_OK;
  if (p->ws) {
    MMF_CUDA(cudaDeviceSynchronize());
    MMF_CUDA(cudaFree(p->ws));
    p->ws = nullptr;
    p->ws_bytes = 0;
  }
  cudaError_t e = cudaMalloc(&p->ws, bytes);
  if (e != cudaSuccess) return fail(MMF_ERR_NOMEM, std::string("workspace cudaMalloc: ") + cudaGetErrorString(e));
  p->ws_bytes = bytes;
  return MMF_OK;
}

// The host-buffer entry points run on the plan's own streams: they get a workspace of their own so that
// they never alias buffers of device-resident calls still in flight on the caller's stream.
static int ensure_host_ws(mmf_plan* p, size_t bytes) {
  if (bytes <= p->host_ws_bytes) return MMF_OK;
  if (p->host_ws) {
    MMF_CUDA(cudaStreamSynchronize(p->streams[0]));
    MMF_CUDA(cudaStreamSynchronize(p->streams[1]));
    MMF_CUDA(cudaFree(p->host_ws));
    p->host_ws = nullptr;
    p->host_ws_bytes = 0;
  }
  cudaError_t e = cudaMalloc(&p->host_ws, bytes);
  if (e != cudaSuccess) return fail(MMF_ERR_NOMEM, std::string("host-path workspace cudaMalloc: ") + cudaGetErrorString(e));
  p->host_ws_bytes = bytes;
  return MMF_OK;
}

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// carve `bytes` out of a bump pointer
static void* carve(unsigned char*& cur, size_t bytes) {
  void* r = cur;
  cur += align_up(bytes, 256);
  return r;
}

// the same bump allocation over offsets: the start of `bytes` at `end`, which moves past them
static size_t ws_take(size_t& end, size_t bytes) {
  const size_t o = end;
  end += align_up(bytes, 256);
  return o;
}

// Descriptors built on the host for one upload: typed arrays appended back to back, each at a multiple of kDescAlign
// bytes, which every descriptor type's alignment divides (8 at most: the doubles of SosPar, the longs of RsClip and
// RmsClip).  A blob appended to another, or copied to device memory aligned to 16, keeps every part aligned.
constexpr size_t kDescAlign = 16;
struct DescBlob {
  std::vector<unsigned char> bytes;
  size_t size() const { return bytes.size(); }
  // appends src[0, n) and returns its offset
  template <typename T>
  size_t put(const T* src, size_t n) {
    static_assert(kDescAlign % alignof(T) == 0, "descriptor type aligned wider than kDescAlign");
    const size_t o = align_up(bytes.size(), kDescAlign);
    bytes.resize(o + n * sizeof(T), 0);
    if (n) std::memcpy(bytes.data() + o, src, n * sizeof(T));
    return o;
  }
  template <typename T>
  size_t put(const std::vector<T>& v) { return put(v.data(), v.size()); }
};

// One ragged launch's descriptors: clips [n], first_item[n + 1]; items: their total (-1: past 2^31 - 1)
struct RaggedParts {
  size_t clips = 0, first = 0;
  int64_t items = 0;
};

// Distinct chunk tables (SosPar) of a batch.  A row's tables depend on its cascade and on its length only through
// the chunk length (sos_par_chunk), so rows of one chunk length share them.
struct SosParSet {
  std::vector<SosPar> pars;
  // index in pars of the tables of cascade `which` (0 or 1), `a`, for rows of T samples; -1 when the kernel takes none
  int index(int which, const SosArgs& a, long T) {
    const int cl = sos_par_chunk(a, T);
    if (cl < 0) return -1;
    int& idx = of_chunk[which][cl];
    SosPar sp;
    if (idx < 0 && sos_par_fill(a, T, &sp)) {
      idx = (int)pars.size();
      pars.push_back(sp);
    }
    return idx;
  }
  std::vector<int> of_chunk[2] = {std::vector<int>(kSosParMaxChunk + 1, -1), std::vector<int>(kSosParMaxChunk + 1, -1)};
};

static int fill_sos(const double* sos, int n_sections, SosArgs* a) {
  if (n_sections < 1 || n_sections > 16) return fail(MMF_ERR_UNSUPPORTED, "n_sections must be in [1, 16]");
  std::memset(a, 0, sizeof(*a));  // (also the padding: the struct is used as a cache key)
  a->n_sections = n_sections;
  for (int s = 0; s < n_sections; ++s)
    for (int k = 0; k < 6; ++k) a->sos[s][k] = sos[6 * s + k] / (k == 3 ? 1.0 : sos[6 * s + 3]);
  double zi[32];
  int padlen = 0;
  if (host_sos_zi(sos, n_sections, zi, &padlen) != 0) return fail(MMF_ERR_INVALID, "singular SOS section");
  for (int s = 0; s < n_sections; ++s) {
    a->zi[s][0] = zi[2 * s];
    a->zi[s][1] = zi[2 * s + 1];
  }
  a->padlen = padlen;
  return MMF_OK;
}

}  // namespace mmf


namespace mmf {

// Tables of the trajectory FFT live in the plan and are rebuilt only when the
// window / FFT size / band edges change.
static int ensure_mod_tables(mmf_plan* p, int win, int nfft, const int* lo, const int* hi, int n_bands) {
  bool same = p->mod_win == win && p->mod_nfft == nfft && p->mod_n_bands == n_bands;
  for (int b = 0; same && b < n_bands; ++b) same = p->mod_lo[b] == lo[b] && p->mod_hi[b] == hi[b];
  if (same) return MMF_OK;
  MMF_CUDA(cudaDeviceSynchronize());
  for (void* d : p->mod_tables) cudaFree(d);
  p->mod_tables.clear();
  p->d_mod_g = nullptr;
  p->mod_g_kp = 0;
  p->d_mod_hann = nullptr;
  p->d_mod_tw1 = p->d_mod_tw2 = nullptr;
  p->d_mod_lo = p->d_mod_hi = nullptr;
  p->mod_n_bands = -1;
  std::vector<float> hann(nfft, 0.0f);
  for (int i = 0; i < win; ++i) hann[i] = (float)(0.5 - 0.5 * std::cos(2.0 * M_PI * (double)i / (double)win));
  StftGeometry g;
  modspec_geometry(nfft, &g);
  std::vector<float2> tw1, tw2;
  if (modspec_fast_supported(nfft)) host_twiddles(nfft, g, tw1, tw2);
  std::vector<int> vlo(16, 0), vhi(16, 0);
  for (int b = 0; b < n_bands; ++b) {
    vlo[b] = lo[b];
    vhi[b] = hi[b];
  }
  cudaError_t e = cudaSuccess;
  upload(e, p->mod_tables, &p->d_mod_hann, hann);
  upload(e, p->mod_tables, &p->d_mod_tw1, tw1);
  upload(e, p->mod_tables, &p->d_mod_tw2, tw2);
  upload(e, p->mod_tables, &p->d_mod_lo, vlo);
  upload(e, p->mod_tables, &p->d_mod_hi, vhi);
  if (e != cudaSuccess) return cuda_fail(e, "uploading modulation-spectrum tables");
  if (modspec_tc_supported(win, nfft) && !(p->cfg.flags & MMF_FLAG_NO_TC_MODSPEC)) {
    std::vector<uint16_t> g;
    modspec_tc_table(win, nfft, g, &p->mod_g_kp);
    upload(e, p->mod_tables, &p->d_mod_g, g);
    if (e != cudaSuccess) return cuda_fail(e, "uploading modulation-spectrum GEMM operand");
  }
  p->mod_win = win;
  p->mod_nfft = nfft;
  p->mod_n_bands = n_bands;
  for (int b = 0; b < 16; ++b) {
    p->mod_lo[b] = vlo[b];
    p->mod_hi[b] = vhi[b];
  }
  return MMF_OK;
}

// the modulation-spectrum geometry that mmf_modspec and the host-buffer bundle accept; band edges are checked when
// band energies are requested
static int validate_modspec(int win, int hop, int nfft, int n_bands, const int* lo, const int* hi, bool bands) {
  if (win < 1 || hop < 1 || nfft < win || nfft < 32 || nfft > 4096 || (nfft & (nfft - 1)))
    return fail(MMF_ERR_UNSUPPORTED, "need 1 <= win <= nfft, nfft a power of two in [32, 4096], hop >= 1");
  if (n_bands < 0 || n_bands > 16) return fail(MMF_ERR_UNSUPPORTED, "n_bands must be in [0, 16]");
  if (!bands) return MMF_OK;
  if (n_bands > 0 && (!lo || !hi)) return fail(MMF_ERR_INVALID, "band edges are NULL");
  for (int b = 0; b < n_bands; ++b)
    if (lo[b] < 0 || hi[b] > nfft / 2 + 1 || lo[b] > hi[b])
      return fail(MMF_ERR_INVALID, "band bin range outside [0, nfft/2+1]");
  return MMF_OK;
}

ModRoute modspec_route(int win, int hop, int nfft, int n_coef, int n_bands, long T, unsigned flags, long n_clips) {
  if (T < win || hop < 1) return ModRoute{kModNone, 0, 0};
  const long n_win = 1 + (T - win) / hop;
  // a kernel that would need more than 2^31 - 1 work items for the batch leaves it to the next one
  auto chunked = [&](ModPath path, long wc) {
    const long n_chunks = (n_win + wc - 1) / wc;
    return wc > 0 && n_clips * n_chunks <= 0x7fffffffL ? ModRoute{path, wc, n_chunks} : ModRoute{kModNone, 0, 0};
  };
  if (!(flags & MMF_FLAG_NO_TC_MODSPEC)) {
    // windowed DFT of 128 trajectory windows at a time as one tcgen05 GEMM (modspec_tc.cu)
    const ModRoute r = chunked(kModTc, modspec_tc_chunk(win, hop, nfft, n_coef, n_bands, T));
    if (r.path != kModNone) return r;
  }
  if (!modspec_fast_supported(nfft)) return ModRoute{kModGeneric, 0, 0};
  const ModRoute r = chunked(kModClip, modspec_clip_chunk(win, hop, nfft, n_coef, n_bands, T));
  return r.path != kModNone ? r : ModRoute{kModFast, 0, 0};
}

// launch route r (modspec_route) for n_clips clips of T frames; vl: a ragged batch of tc / clip work items instead
static int launch_modspec(mmf_plan* p, const ModRoute& r, const float* mfcc, int64_t n_clips, int n_coef, int64_t T,
                          int win, int hop, int nfft, float* mag, float* band, int n_bands, cudaStream_t st,
                          const ModVarlen* vl = nullptr) {
  float* b = n_bands > 0 ? band : nullptr;
  cudaError_t e = cudaSuccess;
  switch (r.path) {
    case kModNone: return MMF_OK;
    case kModTc:
      e = modspec_tc_launch(mfcc, n_clips, n_coef, T, win, hop, nfft, p->d_mod_g, p->mod_g_kp, r.wc, mag, b,
                            p->d_mod_lo, p->d_mod_hi, n_bands, p->sm_count, st, vl);
      if (e != cudaSuccess) return cuda_fail(e, "modspec_tc_kernel launch");
      return MMF_OK;
    case kModClip:
      e = modspec_clip_launch(mfcc, n_clips, n_coef, T, win, hop, nfft, r.wc, p->d_mod_hann, p->d_mod_tw1,
                              p->d_mod_tw2, mag, b, p->d_mod_lo, p->d_mod_hi, n_bands, st, vl);
      break;
    case kModFast:
      e = modspec_fast_launch(mfcc, n_clips, n_coef, T, win, hop, nfft, p->d_mod_hann, p->d_mod_tw1, p->d_mod_tw2, mag,
                              b, p->d_mod_lo, p->d_mod_hi, n_bands, p->sm_count, st);
      break;
    case kModGeneric:
      e = modspec_launch(mfcc, n_clips, n_coef, T, win, hop, nfft, mag, b, p->d_mod_lo, p->d_mod_hi, n_bands, st);
      break;
  }
  if (e != cudaSuccess) return cuda_fail(e, "modspec kernel launch");
  return MMF_OK;
}

static int run_modspec(mmf_plan* p, const float* mfcc, int64_t n_clips, int n_coef, int64_t T, int win, int hop,
                       int nfft, float* mag, float* band, const int* lo, const int* hi, int n_bands, cudaStream_t st) {
  if (T < win) return MMF_OK;
  if (!band) n_bands = 0;
  int rc = ensure_mod_tables(p, win, nfft, lo, hi, n_bands);
  if (rc) return rc;
  const ModRoute r = modspec_route(win, hop, nfft, n_coef, n_bands, T, p->cfg.flags, n_clips);
  return launch_modspec(p, r, mfcc, n_clips, n_coef, T, win, hop, nfft, mag, band, n_bands, st);
}

// ---- stages of mmf_plan_create for the register FFT (host computations only)

// Tables of the mma.sync mel projection (MMF_FLAG_MMA_MEL).  An n-tile is a run of up to 8 consecutive bands (the N
// of mma.m16n8k8); it is cut short when its bands span more than kTileBlocks k-tiles of 8 bins, so that the wide top
// bands do not pile all their blocks on one warp.  Per tile: the k-tiles whose 8x8 block of the filterbank is not all
// zero, and per block the B fragments (b0: k = lane%4, b1: k = lane%4 + 4; n = lane/4) as plain fp32 (split into
// TF32 hi/lo on the fly).
struct MmaMelTables {
  std::vector<float2> bw;
  std::vector<int> pk8, npair = {0}, tile;  // tile[j] = first band | bands << 16
};
static MmaMelTables mma_mel_tables(const std::vector<float>& mel, int n_mels, int F) {
  MmaMelTables t;
  const int kTileBlocks = 8;
  auto wgt = [&](int k, int band) -> float { return (k < F && band < n_mels) ? mel[(size_t)band * F + k] : 0.0f; };
  auto blocks_of = [&](int b0, int nb, std::vector<int>* out) {
    int cnt = 0;
    for (int k8 = 0; k8 < (F + 7) / 8; ++k8) {
      bool any = false;
      for (int k = 8 * k8; k < 8 * k8 + 8 && !any; ++k)
        for (int b = b0; b < b0 + nb && !any; ++b) any = wgt(k, b) != 0.0f;
      if (any) {
        ++cnt;
        if (out) out->push_back(k8);
      }
    }
    return cnt;
  };
  for (int b0 = 0; b0 < n_mels;) {
    int nb = 1;
    while (nb < 8 && b0 + nb < n_mels && blocks_of(b0, nb + 1, nullptr) <= kTileBlocks) ++nb;
    std::vector<int> ks;
    blocks_of(b0, nb, &ks);
    for (int k8 : ks) {
      t.pk8.push_back(k8);
      for (int lane = 0; lane < 32; ++lane) {
        const int g = lane >> 2, t4 = lane & 3;
        const bool own = g < nb;  // columns beyond the tile's bands belong to the next tile
        t.bw.push_back(make_float2(own ? wgt(8 * k8 + t4, b0 + g) : 0.0f, own ? wgt(8 * k8 + t4 + 4, b0 + g) : 0.0f));
      }
    }
    t.tile.push_back(b0 | (nb << 16));
    t.npair.push_back((int)t.pk8.size());
    b0 += nb;
  }
  return t;
}

struct TileGeo {
  int tf = 0, span_bufs = 2, pt_bufs = 2, ctas = 2, threads = 256, mel_mma = 0, ppitch = 0;
  size_t smem = 0;
};

// Tile geometry of the register-FFT kernel (tf = 0: no tile fits).  Preference: the widest tile first (32 frames =
// one frame per lane / two MMA row tiles in the mel phase), then as much double buffering as two CTAs per SM allow
// (<= 113 KB each: 227 KB per SM, 1 KB reserved per CTA); one CTA per SM as the last resort.  `tpf`: threads per
// frame of the 256-thread transform; `n_pairs`, `n_tiles`: sizes of the tensor-core mel tables.
static TileGeo choose_tile_geometry(const mmf_config& c, int tpf, int packed, int lead, int mel_groups, int mg_n,
                                    int n_pairs, int n_tiles) {
  const int fpw = tpf < 32 ? 32 / tpf : 1;  // frames per warp in the FFT phase
  auto pitch_for = [&](int tf) {
    // bin-pair layout: 8-byte words per bin-pair row; = 2 (mod 16) keeps the 32-bit stores of the two
    // thread groups of a warp on disjoint banks (stft_core.cuh: TilePairs)
    if (mel_groups) return std::max(tf, 2) + 2;
    if (packed) {
      // two-frame path: 64-bit stores of (frame, frame+1) pairs by consecutive bins:
      // pitch == 2 (mod 4) keeps them 8-byte aligned and conflict-free per half-warp
      int pp = std::max(tf, 2);
      while (pp % 4 != 2) ++pp;
      return pp;
    }
    int pp = std::max(tf, fpw);
    if (fpw == 1) {
      if ((pp & 1) == 0) ++pp;
    } else {
      pp = (pp + fpw - 1) / fpw * fpw;
      if (((pp / fpw) & 1) == 0) pp += fpw;
    }
    return pp;
  };
  const size_t budget2 = 113 * 1024, budget1 = 226 * 1024;
  static const int kBufChoices[4][2] = {{2, 2}, {1, 2}, {2, 1}, {1, 1}};  // {span_bufs, pt_bufs}
  auto smem_for = [&](int tf, int span_bufs, int pt_bufs, int mel_mma, int threads) {
    const int span = (tf - 1) * c.hop_length + c.n_fft + lead + 3;
    const int alloc = (span + 255) / 256 * 256;
    return stft_smem_bytes(c.n_fft, alloc, span_bufs, pitch_for(tf), pt_bufs, packed,
                           stft_mel_table_bytes(c.n_fft, c.n_mels, mel_mma, n_pairs, n_tiles, mel_groups, mg_n),
                           threads, mel_groups);
  };
  auto fpi_for = [&](int threads) { return (threads / tpf) * (packed ? 2 : 1); };
  // widest tile (then most double buffering) that fits `budget` with CTAs of `threads`
  auto fit = [&](int mel_mma, int threads, size_t budget, TileGeo* g) {
    const int fpi = fpi_for(threads);
    if (fpi < 1 || fpi > 32) return false;
    for (int cand = 32; cand >= 1; cand >>= 1) {
      if (cand < fpi || cand % fpi) continue;
      for (const auto& ch : kBufChoices) {
        const size_t b = smem_for(cand, ch[0], ch[1], mel_mma, threads);
        if (b <= budget) {
          g->tf = cand;
          g->span_bufs = ch[0];
          g->pt_bufs = ch[1];
          g->smem = b;
          g->threads = threads;
          return true;
        }
      }
    }
    return false;
  };
  auto choose = [&](int mel_mma) {
    TileGeo g;
    g.ctas = 2;
    if (fit(mel_mma, 256, budget2, &g)) return g;
    g.ctas = 1;
    // one CTA per SM: 512 threads (16 warps) when the transform groups are whole warps and the
    // tiles still fit, else 256
    TileGeo g512;
    g512.ctas = 1;
    const bool ok512 = c.n_fft >= 1024 && !mel_mma && fit(mel_mma, 512, budget1, &g512);
    const bool ok256 = fit(mel_mma, 256, budget1, &g);
    if (ok512 && (!ok256 || g512.tf >= g.tf) && !std::getenv("MMF_NO_512")) return g512;
    if (!ok256) g.tf = 0;
    return g;
  };
  // The tensor-core mel (MMF_FLAG_MMA_MEL) keeps its B fragments in shared memory: honoured unless
  // that costs tile width or the second CTA per SM (very wide filterbanks).  Default is the sparse
  // FP32 walk: the filterbank is 95-98 % zeros and the split-precision MMA path measured 3-7 %
  // slower on every BASELINE shape (DESIGN.md section 4).
  TileGeo gs = choose(0), gm = choose(1);
  const bool units_fit = n_tiles * 2 <= 8 * 16 && n_tiles <= 255;
  const int mel_mma =
      ((c.flags & MMF_FLAG_MMA_MEL) && units_fit && gm.tf != 0 && gm.tf >= gs.tf && gm.ctas >= gs.ctas) ? 1 : 0;
  TileGeo g = mel_mma ? gm : gs;
  // debugging / tuning overrides
  if (const char* e = std::getenv("MMF_TF")) {
    const int v = std::atoi(e);
    const int fpi = fpi_for(256);
    g.threads = 256;
    if (v >= fpi && v <= 32 && (v & (v - 1)) == 0 && v % fpi == 0) g.tf = v;
    if (const char* e2 = std::getenv("MMF_SPAN_BUFS")) g.span_bufs = std::atoi(e2) == 1 ? 1 : 2;
    if (const char* e3 = std::getenv("MMF_PT_BUFS")) g.pt_bufs = std::atoi(e3) == 1 ? 1 : 2;
    g.smem = smem_for(g.tf, g.span_bufs, g.pt_bufs, mel_mma, 256);
    g.ctas = g.smem <= budget2 ? 2 : 1;
    if (g.smem > budget1) g.tf = 0;
  }
  g.mel_mma = mel_mma;
  g.ppitch = pitch_for(g.tf);
  return g;
}

// Tensor-core mel work list: unit = (n-tile, 16-frame m-tile), cost = blocks of the n-tile (npair[n + 1] -
// npair[n]); longest-processing-time assignment to the 8 warps (each unit is produced by exactly one warp).  Fills
// units[w * 16 + i] with (n | m << 8); false if a warp would get more than 16 units.
static bool assign_mma_units(const std::vector<int>& npair, int tf, std::vector<int>& units_out) {
  const int NT = (int)npair.size() - 1, MT = (tf + 15) / 16;
  std::vector<std::pair<int, int>> units;  // (cost, n | m << 8)
  for (int n = 0; n < NT; ++n)
    for (int m = 0; m < MT; ++m) units.push_back({npair[n + 1] - npair[n], n | (m << 8)});
  std::stable_sort(units.begin(), units.end(),
                   [](const std::pair<int, int>& a, const std::pair<int, int>& b) { return a.first > b.first; });
  long load[8] = {0};
  int cnt[8] = {0};
  for (const auto& u : units) {
    int w = 0;
    for (int i = 1; i < 8; ++i)
      if (load[i] < load[w] || (load[i] == load[w] && cnt[i] < cnt[w])) w = i;
    if (cnt[w] >= 16) return false;
    units_out[w * 16 + cnt[w]++] = u.second;
    load[w] += u.first + 2;  // + epilogue
  }
  return true;
}

// Mel band groups of the mel walk: `workers` contiguous runs of bands, balanced on cost = bins walked + bands
// emitted (smallest achievable maximum, greedy fill under a binary-searched bound).  Returns the first band of each
// worker, padded to 257 entries with n_mels.
static std::vector<int> balance_band_split(const MelSparse& sp, const MelGroups& mg, int mel_groups, int n_mels,
                                           int workers) {
  std::vector<int> split(257, n_mels);
  const int cbin = 7, cband = 48;  // measured: 7 instructions per bin, 29 per segment + 19 per band
  const int cgroup = 14, cseg = 41;  // grouped walk (SASS count): per 4-bin weight group, per segment
  auto group_cost = [&](int a, int b) -> long {  // bands [a, b): segments a..b
    if (mel_groups) return (long)cgroup * (mg.segtab[2 * (b + 1) + 1] - mg.segtab[2 * a + 1]) + (long)cseg * (b - a + 1);
    return cbin * (sp.seg_start[b + 1] - sp.seg_start[a]) + cband * (b - a);
  };
  auto fill = [&](long bound, std::vector<int>* out) {
    int a = 0, used = 0;
    while (a < n_mels) {
      if (used == workers) return false;
      int b = a + 1;
      if (group_cost(a, b) > bound) return false;
      while (b < n_mels && group_cost(a, b + 1) <= bound) ++b;
      if (out) (*out)[used] = a;
      a = b;
      ++used;
    }
    if (out)
      for (int w = used; w < 257; ++w) (*out)[w] = n_mels;
    return true;
  };
  long lo = 0, hi = group_cost(0, n_mels);
  while (lo < hi) {
    const long mid = (lo + hi) / 2;
    if (fill(mid, nullptr)) hi = mid; else lo = mid + 1;
  }
  fill(lo, &split);
  return split;
}
}  // namespace mmf

using namespace mmf;

extern "C" {

int mmf_version(void) { return MMF_VERSION; }
int mmf_abi_sizeof(int32_t which) {
  switch (which) {
    case 0: return (int)sizeof(mmf_config);
    case 1: return (int)sizeof(mmf_change_params);
    case 2: return (int)sizeof(mmf_modspec_params);
    case 3: return (int)sizeof(mmf_resample_clip);
    case 4: return (int)sizeof(mmf_amp_params);
    case 5: return (int)sizeof(mmf_env_params);
    case 6: return (int)sizeof(mmf_out_filter);
    default: return -1;
  }
}
const char* mmf_last_error(void) { return g_err.c_str(); }
int64_t mmf_launch_count(int32_t reset) {
  const long v = g_launches;
  if (reset) g_launches = 0;
  return v;
}

int64_t mmf_num_frames(int64_t n_samples, int32_t n_fft, int32_t hop_length) {
  if (hop_length < 1) return -1;
  const int64_t padded = n_samples + 2 * (int64_t)(n_fft / 2);
  if (padded < n_fft) return 0;
  return 1 + (padded - n_fft) / hop_length;
}

int mmf_host_tables(const mmf_config* cfg, float* window, float* mel, float* dct) {
  int rc = validate_cfg(cfg);
  if (rc) return rc;
  const int F = cfg->n_fft / 2 + 1;
  if (window) {
    std::vector<float> w;
    host_window(cfg->win_length, cfg->n_fft, w);
    std::memcpy(window, w.data(), w.size() * sizeof(float));
  }
  if (mel) {
    std::vector<float> m;
    std::vector<double> mf;
    host_mel_dense(cfg->sample_rate, cfg->n_fft, cfg->n_mels, cfg->fmin, cfg->fmax, m, mf);
    std::memcpy(mel, m.data(), (size_t)cfg->n_mels * F * sizeof(float));
  }
  if (dct) {
    std::vector<float> d;
    host_dct(cfg->n_mfcc, cfg->n_mels, d);
    std::memcpy(dct, d.data(), d.size() * sizeof(float));
  }
  return MMF_OK;
}

int mmf_sos_zi(const double* sos, int32_t n_sections, double* zi, int32_t* padlen) {
  if (!sos || !zi) return fail(MMF_ERR_INVALID, "NULL argument");
  int pl = 0;
  if (host_sos_zi(sos, n_sections, zi, &pl) != 0) return fail(MMF_ERR_INVALID, "bad SOS cascade");
  if (padlen) *padlen = pl;
  return MMF_OK;
}

int mmf_plan_create(mmf_plan** out, const mmf_config* cfg) {
  if (!out) return fail(MMF_ERR_INVALID, "out is NULL");
  *out = nullptr;
  int rc = validate_cfg(cfg);
  if (rc) return rc;
  int ndev = 0;
  cudaError_t ce = cudaGetDeviceCount(&ndev);
  if (ce != cudaSuccess || ndev == 0)
    return fail(MMF_ERR_CUDA, std::string("no CUDA device available (this library has no CPU fallback): ") +
                                  cudaGetErrorString(ce));
  if (cfg->device < 0 || cfg->device >= ndev) return fail(MMF_ERR_INVALID, "device ordinal out of range");
  MMF_CUDA(cudaSetDevice(cfg->device));
  cudaDeviceProp prop;
  MMF_CUDA(cudaGetDeviceProperties(&prop, cfg->device));
  if (prop.major < 10)
    return fail(MMF_ERR_UNSUPPORTED, "this library is built for sm_100a (Blackwell B200) only");

  {
    // stream-ordered scratch (cudaMallocAsync in the resampler, the Hilbert envelope and the generic-n_fft path) stays
    // cached in the device's default pool instead of going back to the driver at every synchronisation: with the
    // default release threshold of 0 the Hilbert envelope of one 10 s clip took 1.1 .. 118 ms from call to call
    static bool pool_set[64] = {};
    if (cfg->device < 64 && !pool_set[cfg->device]) {
      cudaMemPool_t pool;
      if (cudaDeviceGetDefaultMemPool(&pool, cfg->device) == cudaSuccess) {
        uint64_t keep = 1ull << 30;  // up to 1 GiB of freed scratch is kept for reuse
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
      }
      pool_set[cfg->device] = true;
    }
  }
  // every return below releases the plan and all it has allocated, except the final one
  std::unique_ptr<mmf_plan, decltype(&mmf_plan_destroy)> p(new mmf_plan(), mmf_plan_destroy);
  p->cfg = *cfg;
  p->F = cfg->n_fft / 2 + 1;
  p->sm_count = prop.multiProcessorCount;
  // the register FFT covers powers of two in [256, 4096]; every other n_fft librosa accepts goes through the
  // FP32 matrix-product DFT (dft_generic.cu)
  p->generic = (cfg->n_fft < 256 || (cfg->n_fft & (cfg->n_fft - 1))) ? 1 : 0;
  p->packed = (!p->generic && stft_packed_supported(cfg->n_fft) && !(cfg->flags & MMF_FLAG_SCALAR_FFT)) ? 1 : 0;
  p->lead = cfg->preemph != 0.0f ? 2 : 0;

  // ---- constant tables of both transforms
  std::vector<float> window, mel, dct;
  std::vector<double> mel_f;
  host_window(cfg->win_length, cfg->n_fft, window);
  host_mel_dense(cfg->sample_rate, cfg->n_fft, cfg->n_mels, cfg->fmin, cfg->fmax, mel, mel_f);
  MelSparse sp;
  if (!host_mel_sparse(mel, mel_f, cfg->sample_rate, cfg->n_fft, cfg->n_mels, sp))
    return fail(MMF_ERR_UNSUPPORTED, "mel filterbank is not a two-slope (triangular) bank");
  host_dct(cfg->n_mfcc, cfg->n_mels, dct);
  p->nc_pad = cfg->n_mfcc <= 16 ? 16 : (cfg->n_mfcc <= 32 ? 32 : (cfg->n_mfcc <= 64 ? 64 : 128));
  std::vector<float> dct_pad((size_t)cfg->n_mels * p->nc_pad, 0.0f);
  for (int k = 0; k < cfg->n_mfcc; ++k)
    for (int m = 0; m < cfg->n_mels; ++m) dct_pad[(size_t)m * p->nc_pad + k] = dct[(size_t)k * cfg->n_mels + m];
  std::vector<float2> w2(p->F);
  for (int k = 0; k < p->F; ++k) w2[k] = make_float2(sp.w2[2 * k], sp.w2[2 * k + 1]);
  std::vector<float4> dct_bfrag;
  mfcc_mma_bfrag(dct.data(), cfg->n_mfcc, cfg->n_mels, dct_bfrag);
  const char* consts_msg = p->generic ? "uploading plan constants (generic n_fft)" : "uploading plan constants";
  cudaError_t e = cudaSuccess;
  upload(e, p->tables, &p->d_window, window);
  upload(e, p->tables, &p->d_seg, sp.seg_start);
  upload(e, p->tables, &p->d_w2, w2);
  upload(e, p->tables, &p->d_dct, dct_pad);
  upload(e, p->tables, &p->d_dct_bfrag, dct_bfrag);
  if (e != cudaSuccess) return cuda_fail(e, consts_msg);

  if (p->generic) {
    std::vector<float> tab;
    dft_generic_table(cfg->n_fft, window, tab, &p->dft_ld);
    upload(e, p->tables, &p->d_dft_tab, tab);
    if (e != cudaSuccess) return cuda_fail(e, consts_msg);
  } else {
    // grouped mel walk on the bin-pair power tile: the default; MMF_FLAG_MEL_WALK / MMF_FLAG_MMA_MEL select
    // the [bin][frame] tile with the sparse walk / the mma.sync projection
    MelGroups mg;
    host_mel_groups(sp, p->F, cfg->n_mels, mg);
    p->mel_groups = (cfg->flags & (MMF_FLAG_MEL_WALK | MMF_FLAG_MMA_MEL)) ? 0 : 1;
    p->mg_n = mg.n_groups;
    const MmaMelTables mma = mma_mel_tables(mel, cfg->n_mels, p->F);
    const int NT = (int)mma.tile.size();
    p->mma_n_pairs = (int)mma.pk8.size();
    p->mma_n_tiles = NT;
    StftGeometry geo{};
    stft_geometry(cfg->n_fft, p->packed, 256, &geo);
    const TileGeo g = choose_tile_geometry(*cfg, geo.tpf, p->packed, p->lead, p->mel_groups, p->mg_n,
                                           p->mma_n_pairs, NT);
    if (g.tf == 0)
      return fail(MMF_ERR_UNSUPPORTED, "hop_length/n_fft combination needs more shared memory than one SM has");
    p->mel_mma = g.mel_mma;
    p->threads = g.threads;
    p->TF = g.tf;
    p->pt_bufs = g.pt_bufs;
    p->span_bufs = g.span_bufs;
    p->ctas_per_sm = g.ctas;
    p->ppitch = g.ppitch;
    p->smem = g.smem;
    p->mel_tab_bytes =
        stft_mel_table_bytes(cfg->n_fft, cfg->n_mels, p->mel_mma, p->mma_n_pairs, NT, p->mel_groups, p->mg_n);
    stft_geometry(cfg->n_fft, p->packed, p->threads, &geo);

    std::vector<int> mma_units(8 * 16, -1);  // [8 warps][16], -1 terminated
    if (p->mel_mma && !assign_mma_units(mma.npair, p->TF, mma_units))
      return fail(MMF_ERR_UNSUPPORTED, "too many mel tiles per warp");  // cannot happen with units_fit
    // 8 warps * (32 / TF) workers of the mel walk
    const std::vector<int> band_split =
        balance_band_split(sp, mg, p->mel_groups, cfg->n_mels, std::min(256, (p->threads / 32) * (32 / p->TF)));
    std::vector<float2> tw1, tw2;
    host_twiddles(cfg->n_fft, geo, tw1, tw2);

    std::vector<int2> segtab(cfg->n_mels + 2);
    for (int j = 0; j < cfg->n_mels + 2; ++j) segtab[j] = make_int2(mg.segtab[2 * j], mg.segtab[2 * j + 1]);
    std::vector<float4> w4((size_t)2 * mg.n_groups);
    for (size_t i = 0; i < w4.size(); ++i) w4[i] = make_float4(mg.w[4 * i], mg.w[4 * i + 1], mg.w[4 * i + 2], mg.w[4 * i + 3]);
    std::vector<int2> segstep(cfg->n_mels + 3);
    for (int j = 0; j < cfg->n_mels + 3; ++j)  // step in 8-byte tile words: two bin-pair rows per group
      segstep[j] = make_int2(mg.segstep[2 * j], mg.segstep[2 * j + 1] * 2 * p->ppitch);
    upload(e, p->tables, &p->d_mg_seg, segtab);
    upload(e, p->tables, &p->d_mg_w, w4);
    upload(e, p->tables, &p->d_mg_step, segstep);
    if (e != cudaSuccess) return cuda_fail(e, "uploading the grouped mel tables");
    upload(e, p->tables, &p->d_tw1, tw1);
    upload(e, p->tables, &p->d_tw2, tw2);
    upload(e, p->tables, &p->d_band_split, band_split);
    upload(e, p->tables, &p->d_mma_bw, mma.bw);
    upload(e, p->tables, &p->d_mma_pk8, mma.pk8);
    upload(e, p->tables, &p->d_mma_npair, mma.npair);
    upload(e, p->tables, &p->d_mma_tile, mma.tile);
    upload(e, p->tables, &p->d_mma_units, mma_units);
    if (e != cudaSuccess) return cuda_fail(e, consts_msg);
  }

  // mel projection as a tcgen05 GEMM (default where it applies; stft_mel_tc.cu)
  if (!(cfg->flags & (MMF_FLAG_NO_TC_MEL | MMF_FLAG_MEL_WALK | MMF_FLAG_MMA_MEL | MMF_FLAG_SPLIT_SMEM)) &&
      stft_mel_tc_supported(cfg->n_fft, stft_mel_tc_active_bands(mel, cfg->n_mels, p->F), cfg->hop_length, p->lead,
                            p->packed)) {
    std::vector<uint16_t> tab;
    stft_mel_tc_table(mel, cfg->n_mels, p->F, tab);
    upload(e, p->tables, &p->d_mel_tc, tab);
    if (e != cudaSuccess) return cuda_fail(e, "uploading the tensor-core mel operand");
    p->mel_tc_act = stft_mel_tc_active_bands(mel, cfg->n_mels, p->F);
    // thread tau of a frame group holds samples 2 (tau + 16 n2), + 1: n2 selects a run of 32 samples
    p->win_lo = 16;
    p->win_hi = 0;
    for (int n2 = 0; n2 < 16; ++n2)
      for (int i = 32 * n2; i < 32 * n2 + 32; ++i)
        if (window[i] != 0.0f) {
          p->win_lo = std::min(p->win_lo, n2);
          p->win_hi = std::max(p->win_hi, n2 + 1);
        }
    if (p->win_hi <= p->win_lo) p->win_lo = 0, p->win_hi = 16;
  }
  // generic-n_fft plans keep the FP32 DCT kernel
  if ((cfg->flags & MMF_FLAG_TC_DCT) && !(cfg->flags & MMF_FLAG_MMA_DCT) && !p->generic &&
      mfcc_tc_supported(cfg->n_mfcc, cfg->n_mels)) {
    std::vector<uint16_t> tab;
    mfcc_tc_table(dct.data(), cfg->n_mfcc, cfg->n_mels, tab, &p->dct_tc_kp);
    upload(e, p->tables, &p->d_dct_tc, tab);
    if (e != cudaSuccess) return cuda_fail(e, "uploading the tensor-core DCT operand");
  }
  if ((cfg->flags & MMF_FLAG_TC_FFT) && tc_fft_supported(cfg->n_fft, cfg->hop_length, cfg->preemph)) {
    std::vector<uint16_t> btab;
    std::vector<float> twf;
    tc_fft_tables(btab, twf);
    upload(e, p->tables, &p->d_tc_btab, btab);
    upload(e, p->tables, &p->d_tc_tw, twf);
    if (e != cudaSuccess) return cuda_fail(e, "uploading tensor-core transform tables");
  }

  // ---- driver entry point for tensor-map encoding (no link-time libcuda dependency)
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
  if (e == cudaSuccess && qres == cudaDriverEntryPointSuccess) p->encode = (PFN_cuTensorMapEncodeTiled_v12000)fn;
  for (int i = 0; i < 2; ++i) cudaStreamCreateWithFlags(&p->streams[i], cudaStreamNonBlocking);
  *out = p.release();
  return MMF_OK;
}

int mmf_plan_destroy(mmf_plan* p) {
  if (!p) return MMF_OK;
  cudaSetDevice(p->cfg.device);
  cudaDeviceSynchronize();
  for (void* d : p->tables) cudaFree(d);
  for (void* d : p->mod_tables) cudaFree(d);
  cudaFree(p->ws);
  cudaFree(p->host_ws);
  for (cudaStream_t s : p->streams)
    if (s) cudaStreamDestroy(s);
  delete p;
  return MMF_OK;
}

}  // extern "C"

namespace mmf {

// shared body of mmf_stft_power / mmf_logmel.  vl: a variable-length batch (log-mel only, power-of-two n_fft) of
// clips of at most n_samples samples, output rows vl->pitch frames apart
static int run_stft(mmf_plan* p, const float* pcm, int64_t n_clips, int64_t n_samples, int64_t clip_stride,
                    float* power, float* logmel, int* clipmax, cudaStream_t st, const Varlen* vl = nullptr) {
  if (!p) return fail(MMF_ERR_INVALID, "plan is NULL");
  if (!pcm) return fail(MMF_ERR_INVALID, "pcm is NULL");
  if (n_clips < 1 || n_samples < 1) return fail(MMF_ERR_INVALID, "n_clips and n_samples must be positive");
  if (clip_stride < n_samples && n_clips > 1) return fail(MMF_ERR_INVALID, "clip_stride < n_samples");
  if (logmel && !clipmax) return fail(MMF_ERR_INVALID, "clipmax buffer required with logmel");
  const mmf_config& c = p->cfg;
  const int64_t T = mmf_num_frames(n_samples, c.n_fft, c.hop_length);
  if (T < 1) return fail(MMF_ERR_INVALID, "input too short for one frame");
  if (T > 0x7fffffff || n_samples + c.n_fft > 0x7fffffffLL)
    return fail(MMF_ERR_UNSUPPORTED, "clip longer than 2^31 samples");
  MMF_CUDA(cudaSetDevice(c.device));

  if (p->generic) {
    // FP32 matrix-product DFT -> power spectrum in HBM (the caller's buffer, or stream-ordered scratch in clip
    // chunks of <= 1 GiB) -> sparse mel walk + log, one frame per thread
    if (clipmax) {
      cudaError_t e = fill_i32_launch(clipmax, n_clips, (int)0x80800000, st);
      if (e != cudaSuccess) return cuda_fail(e, "clipmax init");
    }
    const size_t per_clip = (size_t)p->F * T * 4;
    const int64_t chunk = power ? n_clips : std::max<int64_t>(1, std::min<int64_t>(n_clips, ((size_t)1 << 30) / per_clip));
    float* scratch = nullptr;
    if (!power) MMF_CUDA(cudaMallocAsync((void**)&scratch, (size_t)chunk * per_clip, st));
    cudaError_t e = cudaSuccess;
    for (int64_t c0 = 0; c0 < n_clips && e == cudaSuccess; c0 += chunk) {
      const int64_t nc = std::min<int64_t>(chunk, n_clips - c0);
      float* pw = power ? power + (size_t)c0 * p->F * T : scratch;
      e = dft_generic_power_launch(pcm + (size_t)c0 * clip_stride, nc, n_samples, clip_stride, (int)T, c.hop_length,
                                   c.n_fft, c.preemph, p->d_dft_tab, p->dft_ld, pw, st);
      if (e == cudaSuccess && logmel)
        e = mel_from_power_launch(pw, nc, p->F, (int)T, c.n_mels, c.amin, p->d_seg, p->d_w2,
                                  logmel + (size_t)c0 * c.n_mels * T, clipmax + c0, st);
    }
    if (scratch) cudaFreeAsync(scratch, st);
    if (e != cudaSuccess) return cuda_fail(e, "generic DFT kernels launch");
    return MMF_OK;
  }

  StftArgs a{};
  a.pcm = pcm;
  a.n_samples = n_samples;
  a.clip_stride = clip_stride;
  a.T = (int)T;
  a.hop = c.hop_length;
  a.TF = p->TF;
  a.tiles_per_clip = (int)((T + p->TF - 1) / p->TF);
  a.n_tiles = (long)a.tiles_per_clip * n_clips;
  a.lead = p->lead;
  a.span_floats = (p->TF - 1) * c.hop_length + c.n_fft + p->lead + 3;  // +3: 16-byte aligned start
  a.span_alloc = (a.span_floats + 255) / 256 * 256;
  a.ppitch = p->ppitch;
  a.pt_bufs = p->pt_bufs;
  a.packed = p->packed;
  a.threads = p->threads;
  a.mel_mma = p->mel_mma;
  a.m_tiles = (p->TF + 15) / 16;
  a.mma_n_pairs = p->mma_n_pairs;
  a.mel_tab_bytes = (int)p->mel_tab_bytes;
  a.mma_bw = p->d_mma_bw;
  a.mma_pk8 = p->d_mma_pk8;
  a.mma_npair = p->d_mma_npair;
  a.mma_tile = p->d_mma_tile;
  a.mma_n_tiles = p->mma_n_tiles;
  a.mma_units = p->d_mma_units;
  a.early_tma = 1;
#ifdef MMF_PROFILE  // profiling builds only: a stray environment variable must never change results
  if (const char* e = std::getenv("MMF_DEBUG_SKIP")) a.debug_skip = std::atoi(e);
  if (const char* e = std::getenv("MMF_EARLY_TMA")) a.early_tma = std::atoi(e);
#endif
  a.span_bufs = p->span_bufs;
  a.vec_ok = (c.hop_length % 2 == 0) ? 1 : 0;
  a.split_regs = (c.n_fft == 512 && !(c.flags & MMF_FLAG_SPLIT_SMEM)) ? 1 : 0;
  a.n_mels = c.n_mels;
  a.amin = c.amin;
  a.preemph = c.preemph;
  a.window = p->d_window;
  a.tw1 = p->d_tw1;
  a.tw2 = p->d_tw2;
  a.seg_start = p->d_seg;
  a.band_split = p->d_band_split;
  a.w2 = p->d_w2;
  a.mel_groups = p->mel_groups;
  a.mg_n = p->mg_n;
  a.mg_seg = p->d_mg_seg;
  a.mg_step = p->d_mg_step;
  a.mg_w = p->d_mg_w;
  a.logmel = logmel;
  a.clipmax = clipmax;
  a.power = power;
  a.pitch = (int)T;
  if (vl) {
    a.n_tiles = vl->n_units;
    a.pitch = vl->pitch;
    a.vl_len = vl->len;
    a.vl_T = vl->T;
    a.vl_first = vl->first;
    a.vl_clips = (int)n_clips;
  }

  // TMA needs a 16-byte aligned base and row pitch; otherwise use the plain loader
  CUtensorMap tmap;
  std::memset(&tmap, 0, sizeof(tmap));
  bool tma = p->encode != nullptr && !(c.flags & MMF_FLAG_NO_TMA) && ((uintptr_t)pcm % 16 == 0) &&
             ((clip_stride * 4) % 16 == 0 || n_clips == 1);
  if (tma) {
    cuuint64_t gdim[2] = {(cuuint64_t)n_samples, (cuuint64_t)n_clips};
    cuuint64_t gstr[1] = {(cuuint64_t)(n_clips == 1 ? align_up((size_t)n_samples * 4, 16) : clip_stride * 4)};
    cuuint32_t box[2] = {256, 1};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = p->encode(&tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)pcm, gdim, gstr, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) tma = false;
  }
  a.use_tma = tma ? 1 : 0;

  if (clipmax) {
    cudaError_t e = fill_i32_launch(clipmax, n_clips, (int)0x80800000, st)  /* key of -FLT_MAX */;
    if (e != cudaSuccess) return cuda_fail(e, "clipmax init");
  }
  // the mel projection on the tensor cores wherever the plan supports it -- a decision of the configuration alone, so
  // that a clip's features never depend on the size or the chunking of the batch it came in
  if (p->d_mel_tc && logmel && !power && (vl || ((T + 127) / 128) * n_clips < 0x7fffffffLL)) {
    cudaError_t e = stft_mel_tc_launch(tmap, tma ? 1 : 0, pcm, n_clips, n_samples, clip_stride, (int)T, c.hop_length, p->lead, c.n_mels, p->mel_tc_act, c.amin,
                                       c.preemph, p->d_window, p->win_lo, p->win_hi, p->d_tw1, p->d_mel_tc, logmel, clipmax, p->sm_count, st, vl);
    count_launch();
    if (e != cudaSuccess) return cuda_fail(e, "stft_mel_tc_kernel launch");
    return MMF_OK;
  }
  const long max_ctas = (long)p->ctas_per_sm * p->sm_count;
  const int grid = (int)std::min<long>(a.n_tiles, max_ctas);
  cudaError_t e = stft_mel_launch(c.n_fft, tmap, a, grid, p->smem, st);
  count_launch();
  if (e != cudaSuccess) return cuda_fail(e, "stft_mel_kernel launch");
  return MMF_OK;
}

// zero-phase IIR over independent rows: chunk-parallel kernel when the extended row fits in
// shared memory (<= 6112 samples, <= 4 sections); super-block scan for long rows; else the
// sequential kernel (many long rows, or more than 4 sections)
static cudaError_t sosfiltfilt_any(const void* x, int x_is_f32, long rows, long T, long xs, int group_rows,
                                   long group_stride, const SosArgs& a, double* y, long ys, cudaStream_t st) {
  SosPar par;
  if (sos_par_fill(a, T, &par))
    return sosfiltfilt_par_launch(x, x_is_f32, rows, T, xs, group_rows, group_stride, par, y, ys, st);
  // long rows, few of them: the sequential kernel would walk every sample one by one
  if (sos_long_supported(a, rows, T) && (size_t)rows * (size_t)(T + 2 * a.padlen) * 8 <= ((size_t)1 << 30))
    return sosfiltfilt_long_launch(x, x_is_f32, rows, T, xs, group_rows, group_stride, a, y, ys, st);
  return sosfiltfilt_launch_grouped(x, x_is_f32, rows, T, xs, group_rows, group_stride, a, y, ys, st);
}

// The K3 (clamp + DCT-II (+ delta)) kernel: a decision of the plan alone.  Tensor-core DCT-II (mma.sync TF32 x3) on
// request only: measured 185 us against 95 us for the FP32 kernel on the bench workload (DESIGN.md section 4).
// MMF_FLAG_TC_DCT: tcgen05 GEMM over 128-frame tiles (mfcc_tc.cu), where the plan built its operand.
enum MfccKernel { kMfccFp32, kMfccMma, kMfccTc };
static MfccKernel mfcc_kernel(const mmf_plan* p) {
  if ((p->cfg.flags & MMF_FLAG_MMA_DCT) && mfcc_mma_supported(p->cfg.n_mfcc, p->cfg.n_mels)) return kMfccMma;
  return p->d_dct_tc ? kMfccTc : kMfccFp32;
}

// kernel k over n_clips clips of T frames, 65535 clips per launch; vT: each clip's own frame count (fp32 kernel only)
static int mfcc_run(const mmf_plan* p, MfccKernel k, float* logmel, const int* clipmax, int64_t n_clips, int64_t T,
                    float* mfcc, float* delta, int clamp_in_place, cudaStream_t st, const int* vT = nullptr) {
  const mmf_config& c = p->cfg;
  for (int64_t c0 = 0; c0 < n_clips; c0 += 65535) {
    const int64_t nc = std::min<int64_t>(65535, n_clips - c0);
    float *lm = logmel + (size_t)c0 * c.n_mels * T, *mf = mfcc + (size_t)c0 * c.n_mfcc * T;
    float* dl = delta ? delta + (size_t)c0 * c.n_mfcc * T : nullptr;
    const cudaError_t e =
        k == kMfccMma ? mfcc_mma_launch(p->d_dct_bfrag, lm, clipmax + c0, nc, T, c.n_mels, c.n_mfcc, c.top_db, mf, dl,
                                        clamp_in_place, st)
        : k == kMfccTc ? mfcc_tc_launch(p->d_dct_tc, p->dct_tc_kp, lm, clipmax + c0, nc, T, c.n_mels, c.n_mfcc,
                                        c.top_db, mf, dl, clamp_in_place, p->sm_count, st)
                       : mfcc_launch(p->d_dct, p->nc_pad, lm, clipmax + c0, nc, T, c.n_mels, c.n_mfcc, c.top_db, mf,
                                     dl, clamp_in_place, st, vT ? vT + c0 : nullptr);
    if (e != cudaSuccess)
      return cuda_fail(e, k == kMfccTc ? "mfcc_tc_kernel launch"
                          : vT ? "mfcc_kernel (variable-length) launch" : "mfcc_kernel launch");
  }
  return MMF_OK;
}

}  // namespace mmf

extern "C" {

int mmf_stft_power(mmf_plan* plan, const float* pcm_dev, int64_t n_clips, int64_t n_samples, int64_t clip_stride,
                   float* power_dev, void* stream) {
  if (!power_dev) return fail(MMF_ERR_INVALID, "power_dev is NULL");
  if (plan && plan->d_tc_btab && pcm_dev && n_clips >= 1 && n_samples >= 1 && (clip_stride >= n_samples || n_clips == 1)) {
    // tcgen05 transform (MMF_FLAG_TC_FFT): fp16 x3 GEMM stages, accumulators in tensor memory
    const int64_t T = mmf_num_frames(n_samples, plan->cfg.n_fft, plan->cfg.hop_length);
    if (T >= 1 && T <= 0x7fffffff) {
      MMF_CUDA(cudaSetDevice(plan->cfg.device));
      cudaError_t e = tc_fft_power_launch(pcm_dev, n_clips, n_samples, clip_stride, (int)T, plan->cfg.hop_length,
                                          plan->d_window, plan->d_tc_btab, plan->d_tc_tw, power_dev, plan->sm_count,
                                          (cudaStream_t)stream);
      if (e != cudaSuccess) return cuda_fail(e, "tc_fft512_kernel launch");
      return MMF_OK;
    }
  }
  return run_stft(plan, pcm_dev, n_clips, n_samples, clip_stride, power_dev, nullptr, nullptr, (cudaStream_t)stream);
}

int mmf_logmel(mmf_plan* plan, const float* pcm_dev, int64_t n_clips, int64_t n_samples, int64_t clip_stride,
               float* logmel_dev, int32_t* clipmax_dev, void* stream) {
  if (!logmel_dev) return fail(MMF_ERR_INVALID, "logmel_dev is NULL");
  return run_stft(plan, pcm_dev, n_clips, n_samples, clip_stride, nullptr, logmel_dev, clipmax_dev,
                  (cudaStream_t)stream);
}

int mmf_mfcc(mmf_plan* plan, float* logmel_dev, const int32_t* clipmax_dev, int64_t n_clips, int64_t T,
             float* mfcc_dev, float* delta_dev, int32_t clamp_in_place, void* stream) {
  if (!plan || !logmel_dev || !clipmax_dev || !mfcc_dev) return fail(MMF_ERR_INVALID, "NULL argument");
  if (n_clips < 1 || T < 1) return fail(MMF_ERR_INVALID, "n_clips and T must be positive");
  MMF_CUDA(cudaSetDevice(plan->cfg.device));
  return mfcc_run(plan, mfcc_kernel(plan), logmel_dev, clipmax_dev, n_clips, T, mfcc_dev, delta_dev, clamp_in_place,
                  (cudaStream_t)stream);
}

int mmf_sosfiltfilt(mmf_plan* plan, const void* x_dev, int32_t x_is_f32, int64_t rows, int64_t T,
                    int64_t x_row_stride, const double* sos_host, int32_t n_sections, double* y_dev,
                    int64_t y_row_stride, void* stream) {
  if (!plan || !x_dev || !sos_host || !y_dev) return fail(MMF_ERR_INVALID, "NULL argument");
  if (rows < 1) return fail(MMF_ERR_INVALID, "rows must be positive");
  SosArgs a;
  int rc = fill_sos(sos_host, n_sections, &a);
  if (rc) return rc;
  if (T <= a.padlen) return too_short(a.padlen);
  MMF_CUDA(cudaSetDevice(plan->cfg.device));
  cudaError_t e = sosfiltfilt_any(x_dev, x_is_f32, rows, T, x_row_stride,
                                  (int)(rows > 0x7fffffffL ? 0x7fffffff : rows), 0, a, y_dev, y_row_stride,
                                  (cudaStream_t)stream);
  if (e != cudaSuccess) return cuda_fail(e, "sosfiltfilt_kernel launch");
  return MMF_OK;
}

int mmf_delta_norm(mmf_plan* plan, const double* x_dev, int64_t n_clips, int32_t rows_per_clip, int64_t T,
                   int32_t method, double* tot_dev, void* stream) {
  if (!plan || !x_dev || !tot_dev) return fail(MMF_ERR_INVALID, "NULL argument");
  if (n_clips < 1 || rows_per_clip < 1 || T < 1) return fail(MMF_ERR_INVALID, "sizes must be positive");
  MMF_CUDA(cudaSetDevice(plan->cfg.device));
  for (int64_t c0 = 0; c0 < n_clips; c0 += 65535) {
    const int64_t nc = std::min<int64_t>(65535, n_clips - c0);
    cudaError_t e = delta_norm_launch(x_dev + (size_t)c0 * rows_per_clip * T, nc, rows_per_clip, T, method,
                                      tot_dev + (size_t)c0 * T, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(e, "delta_norm_kernel launch");
  }
  return MMF_OK;
}

int mmf_modspec(mmf_plan* plan, const float* mfcc_dev, int64_t n_clips, int32_t n_coef, int64_t T, int32_t win,
                int32_t hop, int32_t nfft, float* mag_dev, float* band_dev, const int32_t* band_lo_host,
                const int32_t* band_hi_host, int32_t n_bands, void* stream) {
  if (!plan || !mfcc_dev) return fail(MMF_ERR_INVALID, "NULL argument");
  int rc = validate_modspec(win, hop, nfft, n_bands, band_lo_host, band_hi_host, band_dev != nullptr);
  if (rc) return rc;
  if (n_clips < 1 || n_coef < 1) return fail(MMF_ERR_INVALID, "n_clips and n_coef must be positive");
  MMF_CUDA(cudaSetDevice(plan->cfg.device));
  return run_modspec(plan, mfcc_dev, n_clips, n_coef, T, win, hop, nfft, mag_dev, band_dev, band_lo_host, band_hi_host,
                     n_bands, (cudaStream_t)stream);
}

}  // extern "C"

namespace mmf {

// Host half of a variable-length K6 batch (mmf_modspec_varlen): each clip's route and the compacted work items, and
// the layout of the workspace the run step carves from.  Clip i has T[i] <= pitch frames.
struct ModspecVarlen {
  int64_t n_clips = 0, W = 0;  // W: windows per output row, the most of any clip
  int nbe = 0, nb = 0;         // band outputs actually written; bins per window
  std::vector<int64_t> T;  // frames of each clip
  std::vector<ModRoute> route;
  std::vector<int> n_win;
  long n_items[2] = {0, 0}, wc_max[2] = {0, 0};  // [0] tc, [1] clip
  std::vector<int64_t> single;                   // clips on the fast / generic kernel
  std::vector<ModItem> items;
  bool tails = false;
  DescBlob desc;  // the descriptors, at the workspace start: work items and window counts
  size_t o_items = 0, o_nwin = 0, o_single = 0, bytes = 0;  // workspace layout (bytes: all of it)
};

// W of a batch, checking every T[i] in [0, pitch] (no plan or device needed)
static int modspec_varlen_windows(const int64_t* T_host, int64_t n_clips, int64_t pitch, int win, int hop, int64_t* W) {
  *W = 0;
  for (int64_t i = 0; i < n_clips; ++i) {
    const int64_t T = T_host[i];
    if (T < 0 || T > pitch) {
      char buf[160];
      std::snprintf(buf, sizeof(buf), "clip %lld: T %lld must be in [0, pitch = %lld]", (long long)i, (long long)T,
                    (long long)pitch);
      return fail(MMF_ERR_INVALID, buf);
    }
    if (T >= win) *W = std::max<int64_t>(*W, 1 + (T - win) / hop);
  }
  return MMF_OK;
}

// routing (host only): each clip as its own call, the tc / clip kernels' chunks as work items.  W > 0.
static int modspec_varlen_route(unsigned flags, const int64_t* T_host, int64_t n_clips, int n_coef, int64_t W, int win,
                                int hop, int nfft, int nbe, bool want_mag, ModspecVarlen& v) {
  v.n_clips = n_clips;
  v.W = W;
  v.nbe = nbe;
  v.nb = nfft / 2 + 1;
  v.T.assign(T_host, T_host + n_clips);
  v.route.assign((size_t)n_clips, ModRoute{});
  v.n_win.assign((size_t)n_clips, 0);
  for (int64_t i = 0; i < n_clips; ++i) {
    const ModRoute r = modspec_route(win, hop, nfft, n_coef, nbe, T_host[i], flags);
    v.route[i] = r;
    v.n_win[i] = T_host[i] >= win ? (int)(1 + (T_host[i] - win) / hop) : 0;
    v.tails |= v.n_win[i] < W;
    if (r.path == kModTc || r.path == kModClip) {
      const int k = r.path == kModTc ? 0 : 1;
      v.n_items[k] += r.n_chunks;
      v.wc_max[k] = std::max(v.wc_max[k], r.wc);
    } else if (r.path != kModNone) {
      v.single.push_back(i);
    }
  }
  if (v.n_items[0] > 0x7fffffffL || v.n_items[1] > 0x7fffffffL)
    return fail(MMF_ERR_UNSUPPORTED, "variable-length batch of more than 2^31 - 1 modulation-spectrum work items");
  v.items.resize((size_t)(v.n_items[0] + v.n_items[1]));
  size_t at[2] = {0, (size_t)v.n_items[0]};
  for (int64_t i = 0; i < n_clips; ++i) {
    const ModRoute& r = v.route[i];
    if (r.path != kModTc && r.path != kModClip) continue;
    size_t& k = at[r.path == kModTc ? 0 : 1];
    for (long c = 0; c < r.n_chunks; ++c) {
      const long w0 = c * r.wc;
      v.items[k++] = ModItem{(int)i, (int)w0, (int)std::min<long>(r.wc, v.n_win[i] - w0), v.n_win[i]};
    }
  }
  // workspace: the descriptors, then the single-clip region (input rows, magnitudes)
  v.o_items = v.desc.put(v.items);
  v.o_nwin = v.desc.put(v.n_win);
  v.o_single = align_up(v.desc.size(), 256);
  size_t single_bytes = 0;
  for (int64_t i : v.single)
    single_bytes = std::max(single_bytes, align_up((size_t)n_coef * T_host[i] * 4, 256) +
                                              (want_mag ? (size_t)n_coef * v.n_win[i] * v.nb * 4 : 0));
  v.bytes = v.o_single + single_bytes;
  return MMF_OK;
}

// device half: launches the batch routed by v on `st`, carving from `base` (v.bytes).  `dd`: v.desc already on the
// device (null: uploaded to `base` here, a copy that waits for the stream).  The modulation tables must be current
// (ensure_mod_tables).
static int modspec_varlen_run(mmf_plan* plan, const ModspecVarlen& v, unsigned char* base, const unsigned char* dd,
                              const float* mfcc_dev, int n_coef, int64_t pitch, int win, int hop, int nfft,
                              float* mag_dev, float* band_dev, cudaStream_t st) {
  int rc;
  const int64_t n_clips = v.n_clips, W = v.W;
  const int nbe = v.nbe, nb = v.nb;
  if (!dd) {
    MMF_CUDA(cudaMemcpyAsync(base, v.desc.bytes.data(), v.desc.size(), cudaMemcpyHostToDevice, st));
    dd = base;
  }

  // ---- the batched clips: one launch per kernel
  for (int k = 0; k < 2; ++k) {
    if (!v.n_items[k]) continue;
    const ModVarlen vl{(const ModItem*)(dd + v.o_items) + (k ? v.n_items[0] : 0), v.n_items[k], (long)W,
                       (int)v.wc_max[k]};
    const ModRoute r{k ? kModClip : kModTc, v.wc_max[k], 0};
    if ((rc = launch_modspec(plan, r, mfcc_dev, n_clips, n_coef, pitch, win, hop, nfft, mag_dev, band_dev, nbe, st,
                             &vl)))
      return rc;
  }

  // ---- the other clips: the single-clip call on contiguous rows, copied into the padded rows
  for (int64_t i : v.single) {
    const size_t Ti = (size_t)v.T[i], wi = (size_t)v.n_win[i];
    float* x1 = (float*)(base + v.o_single);
    float* mag1 = mag_dev ? (float*)(base + v.o_single + align_up((size_t)n_coef * Ti * 4, 256)) : nullptr;
    MMF_CUDA(cudaMemcpy2DAsync(x1, Ti * 4, mfcc_dev + (size_t)i * n_coef * pitch, (size_t)pitch * 4, Ti * 4,
                               (size_t)n_coef, cudaMemcpyDeviceToDevice, st));
    // a clip's band rows [n_win_i, n_bands] are the start of its padded rows [W, n_bands]: written in place
    float* band1 = nbe > 0 ? band_dev + (size_t)i * W * nbe : nullptr;
    if ((rc = launch_modspec(plan, v.route[i], x1, 1, n_coef, (int64_t)Ti, win, hop, nfft, mag1, band1, nbe, st)))
      return rc;
    if (mag1)
      MMF_CUDA(cudaMemcpy2DAsync(mag_dev + (size_t)i * n_coef * W * nb, (size_t)W * nb * 4, mag1, wi * nb * 4,
                                 wi * nb * 4, (size_t)n_coef, cudaMemcpyDeviceToDevice, st));
  }
  if (v.tails && (mag_dev || nbe > 0)) {
    cudaError_t e = modspec_tails_launch((long)n_clips, (const int*)(dd + v.o_nwin), (long)W, mag_dev, n_coef, nb,
                                         nbe > 0 ? band_dev : nullptr, nbe, st);
    if (e != cudaSuccess) return cuda_fail(e, "modspec_tails_kernel launch");
  }
  return MMF_OK;
}

}  // namespace mmf

extern "C" {

// Variable-length batch.  Each clip takes the route and the chunking its own mmf_modspec call would take
// (modspec_route) -- which is what makes its outputs bit-identical to that call.  Clips on the tcgen05 and the
// clip-resident kernel run in one launch per kernel for the whole batch, as a compacted list of (clip, chunk) work
// items; clips on the fast or the generic kernel run one by one through workspace and are copied into their padded
// rows.  One launch then zeroes every window past a clip's own.
int mmf_modspec_varlen(mmf_plan* plan, const float* mfcc_dev, int64_t n_clips, int32_t n_coef, const int64_t* T_host,
                       int64_t pitch, int32_t win, int32_t hop, int32_t nfft, float* mag_dev, float* band_dev,
                       const int32_t* band_lo_host, const int32_t* band_hi_host, int32_t n_bands, void* stream) {
  using namespace mmf;
  // the geometry and the lengths first: these checks need neither a plan nor a device
  int rc = validate_modspec(win, hop, nfft, n_bands, band_lo_host, band_hi_host, band_dev != nullptr);
  if (rc) return rc;
  if (!T_host) return fail(MMF_ERR_INVALID, "T_host is NULL");
  if (n_clips < 1 || n_coef < 1) return fail(MMF_ERR_INVALID, "n_clips and n_coef must be positive");
  if (n_clips > 0x7fffffff) return fail(MMF_ERR_UNSUPPORTED, "more than 2^31 - 1 clips");
  int64_t W = 0;  // windows per output row: the most of any clip
  if ((rc = modspec_varlen_windows(T_host, n_clips, pitch, win, hop, &W))) return rc;
  if (!plan || !mfcc_dev) return fail(MMF_ERR_INVALID, "NULL argument");
  if (W > 0x7fffffff) return fail(MMF_ERR_UNSUPPORTED, "more than 2^31 - 1 windows per clip");
  if (W == 0) return MMF_OK;  // no clip reaches a window: nothing to compute or zero

  const int nbe = band_dev ? n_bands : 0;  // band outputs actually written
  ModspecVarlen v;
  if ((rc = modspec_varlen_route((unsigned)plan->cfg.flags, T_host, n_clips, n_coef, W, win, hop, nfft, nbe,
                                 mag_dev != nullptr, v)))
    return rc;
  MMF_CUDA(cudaSetDevice(plan->cfg.device));
  if ((rc = ensure_mod_tables(plan, win, nfft, band_lo_host, band_hi_host, nbe))) return rc;
  if ((rc = ensure_ws(plan, (64 << 10) + v.bytes))) return rc;
  return modspec_varlen_run(plan, v, (unsigned char*)plan->ws + (64 << 10), nullptr, mfcc_dev, n_coef, pitch, win, hop,
                            nfft, mag_dev, band_dev, (cudaStream_t)stream);
}

}  // extern "C"

namespace mmf {

static size_t change_ws_bytes(const mmf_plan* p, int64_t n_clips, int64_t T, bool need_logmel, bool need_mfcc,
                              int rows) {
  size_t b = 64 << 10;
  if (need_logmel) b += align_up((size_t)n_clips * p->cfg.n_mels * T * 4, 256);
  b += align_up((size_t)n_clips * 4, 256);
  if (need_mfcc) b += align_up((size_t)n_clips * p->cfg.n_mfcc * T * 4, 256);
  b += align_up((size_t)n_clips * rows * T * 8, 256);
  b += align_up((size_t)n_clips * T * 8, 256);
  return b;
}

// Route of the stage after the log-mel: K3 folded into the fused kernel (FROM_LM), the K3 kernel then the fused kernel,
// or the K3 kernel then separate filter and derivative + norm kernels.  smem: the fused kernel's shared memory.
enum ChangePath { kChangeFolded, kChangeFused, kChangeUnfused };
struct ChangeRoute { ChangePath path; MfccKernel k3; size_t smem; };

// One kernel per clip from log-mel to the curve: clamp + DCT-II feed the float64 row buffers in shared memory directly;
// MFCC / delta go to HBM only if the caller asked for them.  Measured on the bench workload: 1 % faster than the
// separate MFCC kernel without a delta output, 1 % slower with one when the modulation spectrum follows (DESIGN.md
// section 4) -- hence the default.  The fused kernel's DCT phase takes up to kFusedNC coefficients.
static bool change_folds(const mmf_plan* p, bool want_delta) {
  const unsigned f = (unsigned)p->cfg.flags;
  return ((f & MMF_FLAG_FOLD_MFCC) || !want_delta) && !(f & (MMF_FLAG_SEPARATE_MFCC | MMF_FLAG_MMA_DCT)) &&
         p->cfg.n_mfcc <= kFusedNC;
}

// Batches: the output filter of the curve runs as its own launch (one warp per clip, all clips at once) instead of on
// ONE warp of the per-clip CTA while its other 11 wait (27 % of that kernel's stall samples, ncu round 2); the raw
// curve makes an 8 KB round trip per clip.  Same routine on the same buffer contents: bit-identical.
static bool change_split_out(bool out_iir, int64_t n_clips) { return out_iir && n_clips >= 32; }

// The route of n_clips clips of T frames, for run_post and for each clip of a variable-length batch.  pa / po: the row
// and (out_iir) output filter's chunk tables at T, null where the chunk-parallel kernel does not take the row.
static ChangeRoute change_route(const mmf_plan* p, bool want_delta, int first, int rows, int64_t T, bool out_iir,
                                const SosPar* pa, const SosPar* po, int64_t n_clips) {
  const mmf_config& c = p->cfg;
  ChangeRoute r{kChangeUnfused, mfcc_kernel(p), 0};
  if ((c.flags & MMF_FLAG_UNFUSED_CHANGE) || !pa || (out_iir && !po)) return r;
  const SosPar* a2 = out_iir ? po : nullptr;
  const bool split = change_split_out(out_iir, n_clips);
  if (change_folds(p, want_delta) && n_clips <= 0x7fffffff &&
      change_fused_lm_supported(*pa, a2, split, c.n_mfcc, c.n_mels, first, rows, T, &r.smem))
    r.path = kChangeFolded;
  else if (change_fused_supported(*pa, a2, split, rows, T, &r.smem))
    r.path = kChangeFused;
  return r;
}

// log-mel -> clamp -> MFCC (+delta) -> zero-phase Butterworth per coefficient ->
// derivative + norm -> output filter.  `cur` bumps through caller-provided workspace.
static int run_post(mmf_plan* p, unsigned char*& cur, float* logmel, const int* clipmax, int64_t n_clips, int64_t T,
                    const mmf_change_params* prm, double* tot, float* mfcc_out, float* delta_out, int clamp_in_place,
                    cudaStream_t st) {
  const mmf_config& c = p->cfg;
  const int first = prm->remove_first ? 1 : 0;
  const int rows = c.n_mfcc - first;
  if (rows < 1) return fail(MMF_ERR_INVALID, "removeFirst leaves no MFCC rows");
  SosArgs sa, so;
  int rc = fill_sos(prm->sos, prm->n_sections, &sa);
  if (rc) return rc;
  const bool out_iir = prm->out_kind == 0;
  if (out_iir && (rc = fill_sos(prm->out_sos, prm->out_n_sections, &so))) return rc;
  if (T <= sa.padlen) return too_short(sa.padlen);
  if (out_iir && T <= so.padlen) return too_short(so.padlen);
  SosPar pa, po;
  const bool has_pa = sos_par_fill(sa, T, &pa), has_po = out_iir && sos_par_fill(so, T, &po);
  const ChangeRoute r = change_route(p, delta_out != nullptr, first, rows, T, out_iir, has_pa ? &pa : nullptr,
                                     has_po ? &po : nullptr, n_clips);
  float* mfcc = nullptr;
  if (r.path != kChangeFolded) {
    mfcc = mfcc_out ? mfcc_out : (float*)carve(cur, (size_t)n_clips * c.n_mfcc * T * 4);
    if ((rc = mfcc_run(p, r.k3, logmel, clipmax, n_clips, T, mfcc, delta_out, clamp_in_place, st))) return rc;
  }
  if (r.path != kChangeUnfused) {
    // fused per-clip kernel: row filters, derivative + norm and the output filter with the
    // float64 rows resident in shared memory (script/mfcc.py:393-425)
    const bool folded = r.path == kChangeFolded, split_out = change_split_out(out_iir, n_clips);
    const FusedMfccArgs lm{p->d_dct, p->nc_pad, logmel, clipmax, c.n_mels, c.top_db, mfcc_out, delta_out,
                           clamp_in_place};
    double* raw = split_out ? (double*)carve(cur, (size_t)n_clips * T * 8) : nullptr;
    cudaError_t e = change_fused_launch(mfcc, n_clips, c.n_mfcc, first, rows, T, prm->diff_method, pa,
                                        out_iir ? po : pa, split_out ? 1 : prm->out_kind, split_out ? raw : tot, r.smem,
                                        folded ? &lm : nullptr, st);
    if (e == cudaSuccess && split_out) e = sosfiltfilt_par_launch(raw, 0, n_clips, T, T, 1, T, po, tot, T, st);
    if (e != cudaSuccess)
      return cuda_fail(e, folded ? "change_fused_kernel (from log-mel) launch" : "change_fused_kernel launch");
    return MMF_OK;
  }
  double* filt = (double*)carve(cur, (size_t)n_clips * rows * T * 8);
  double* raw = (double*)carve(cur, (size_t)n_clips * T * 8);
  // Butterworth zero-phase low-pass of rows first..n_mfcc-1 of every clip (script/mfcc.py:398-402)
  cudaError_t e = sosfiltfilt_any(mfcc + (size_t)first * T, 1, n_clips * rows, T, T, rows, (long)c.n_mfcc * T, sa,
                                  filt, T, st);
  if (e != cudaSuccess) return cuda_fail(e, "sosfiltfilt (mfcc rows)");
  double* change = out_iir ? raw : tot;
  if ((rc = mmf_delta_norm(p, filt, n_clips, rows, T, prm->diff_method, change, st))) return rc;
  if (out_iir) {
    e = sosfiltfilt_any(raw, 0, n_clips, T, T, (int)std::min<int64_t>(n_clips, 0x7fffffff), 0, so, tot, T, st);
    if (e != cudaSuccess) return cuda_fail(e, "sosfiltfilt (total change)");
  }
  return MMF_OK;
}

// device-resident body; `base` is a workspace of change_ws_bytes()
static int run_change(mmf_plan* p, unsigned char* base, const float* pcm, int64_t n_clips, int64_t n_samples,
                      int64_t clip_stride, const mmf_change_params* prm, double* tot, float* logmel_out,
                      float* mfcc_out, float* delta_out, cudaStream_t st) {
  const mmf_config& c = p->cfg;
  const int64_t T = mmf_num_frames(n_samples, c.n_fft, c.hop_length);
  unsigned char* cur = base + (64 << 10);
  float* logmel = logmel_out ? logmel_out : (float*)carve(cur, (size_t)n_clips * c.n_mels * T * 4);
  int* clipmax = (int*)carve(cur, (size_t)n_clips * 4);
  int rc;
  if ((rc = run_stft(p, pcm, n_clips, n_samples, clip_stride, nullptr, logmel, clipmax, st))) return rc;
  return run_post(p, cur, logmel, clipmax, n_clips, T, prm, tot, mfcc_out, delta_out, logmel_out ? 1 : 0, st);
}

}  // namespace mmf

extern "C" {

int mmf_mfcc_change(mmf_plan* plan, const float* pcm_dev, int64_t n_clips, int64_t n_samples, int64_t clip_stride,
                    const mmf_change_params* prm, double* tot_dev, float* logmel_dev, float* mfcc_dev,
                    float* delta_dev, void* stream) {
  if (!plan || !pcm_dev || !prm || !tot_dev) return fail(MMF_ERR_INVALID, "NULL argument");
  if (n_clips < 1 || n_samples < 1) return fail(MMF_ERR_INVALID, "n_clips and n_samples must be positive");
  MMF_CUDA(cudaSetDevice(plan->cfg.device));
  const int64_t T = mmf_num_frames(n_samples, plan->cfg.n_fft, plan->cfg.hop_length);
  const int rows = plan->cfg.n_mfcc - (prm->remove_first ? 1 : 0);
  const size_t need = change_ws_bytes(plan, n_clips, T, logmel_dev == nullptr, mfcc_dev == nullptr, std::max(rows, 1));
  int rc = ensure_ws(plan, need);
  if (rc) return rc;
  return run_change(plan, (unsigned char*)plan->ws, pcm_dev, n_clips, n_samples, clip_stride, prm, tot_dev,
                    logmel_dev, mfcc_dev, delta_dev, (cudaStream_t)stream);
}

int mmf_change_from_logmel(mmf_plan* plan, float* logmel_dev, const int32_t* clipmax_dev, int64_t n_clips, int64_t T,
                           const mmf_change_params* prm, double* tot_dev, float* mfcc_dev, float* delta_dev,
                           int32_t clamp_in_place, void* stream) {
  if (!plan || !logmel_dev || !clipmax_dev || !prm || !tot_dev) return fail(MMF_ERR_INVALID, "NULL argument");
  if (n_clips < 1 || T < 1) return fail(MMF_ERR_INVALID, "n_clips and T must be positive");
  MMF_CUDA(cudaSetDevice(plan->cfg.device));
  const int rows = plan->cfg.n_mfcc - (prm->remove_first ? 1 : 0);
  const size_t need = change_ws_bytes(plan, n_clips, T, false, mfcc_dev == nullptr, std::max(rows, 1));
  int rc = ensure_ws(plan, need);
  if (rc) return rc;
  unsigned char* cur = (unsigned char*)plan->ws + (64 << 10);
  return run_post(plan, cur, logmel_dev, clipmax_dev, n_clips, T, prm, tot_dev, mfcc_dev, delta_dev, clamp_in_place,
                  (cudaStream_t)stream);
}

}  // extern "C"

namespace mmf {

// Host half of a variable-length MFCC-change batch (mmf_mfcc_change_varlen): every clip's route, the chunk tables of
// the batched clips, and the layout of the workspace the run step carves from.  Which optional outputs the caller
// wants is part of the routing (a delta output keeps clamp + DCT-II out of the fused kernel, as in the solo call).
struct ChangeVarlen {
  int64_t n_clips = 0;
  int pitch = 0;  // frames per output row: the longest clip's T
  int first = 0, rows = 0;
  bool split_out = false;
  ChangePath path = kChangeFolded;  // the batched clips' route: folded, or the FP32 K3 kernel and the fused kernel
  std::vector<int64_t> len;
  std::vector<int> T_all, T_k1, clips;
  std::vector<int2> pidx;
  std::vector<unsigned> first_unit;
  std::vector<int64_t> fallback;  // clips on the single-clip path
  SosParSet tables;               // row filter (cascade 0) and output filter (cascade 1)
  int i1 = -1, i2 = -1;           // the longest batched clip's tables: they size the launches' shared memory
  size_t fsmem = 0;
  DescBlob desc;  // the descriptors, at the workspace start
  size_t o_len = 0, o_tall = 0, o_tk1 = 0, o_first = 0, o_clips = 0, o_pidx = 0, o_pars = 0;
  size_t o_logmel = 0, o_clipmax = 0, o_mfcc = 0, o_raw = 0, o_single = 0, bytes = 0;  // workspace (bytes: all of it)
};

// Routing (host only).  The lengths are in [1, 2^31 - n_fft); `index_base` is added to the clip index that a
// too-short error names.
static int change_varlen_route(const mmf_plan* plan, int64_t n_clips, const int64_t* n_samples_host,
                               const mmf_change_params* prm, bool want_logmel, bool want_mfcc, bool want_delta,
                               int64_t index_base, ChangeVarlen& v) {
  const mmf_config& c = plan->cfg;
  int64_t n_max = 0;
  for (int64_t i = 0; i < n_clips; ++i) n_max = std::max(n_max, n_samples_host[i]);
  if (n_max + c.n_fft > 0x7fffffffLL) return fail(MMF_ERR_UNSUPPORTED, "clip longer than 2^31 samples");
  v.n_clips = n_clips;
  v.len.assign(n_samples_host, n_samples_host + n_clips);
  v.first = prm->remove_first ? 1 : 0;
  const int first = v.first;
  const int rows = v.rows = c.n_mfcc - first;
  if (rows < 1) return fail(MMF_ERR_INVALID, "removeFirst leaves no MFCC rows");
  SosArgs sa, so;
  int rc = fill_sos(prm->sos, prm->n_sections, &sa);
  if (rc) return rc;
  const bool out_iir = prm->out_kind == 0;
  if (out_iir && (rc = fill_sos(prm->out_sos, prm->out_n_sections, &so))) return rc;
  v.pitch = (int)mmf_num_frames(n_max, c.n_fft, c.hop_length);
  v.T_all.assign((size_t)n_clips, 0);
  for (int64_t i = 0; i < n_clips; ++i) {
    v.T_all[i] = (int)mmf_num_frames(n_samples_host[i], c.n_fft, c.hop_length);
    const int padlen = std::max(sa.padlen, out_iir ? so.padlen : 0);
    if (v.T_all[i] <= padlen) return too_short(v.T_all[i] <= sa.padlen ? sa.padlen : so.padlen, index_base + i);
  }

  // Each clip is routed as its own single-clip call.  The batch takes the clips whose route is its path: folded when
  // the call folds, else the FP32 K3 kernel (the one that takes per-clip frame counts) and the fused kernel.
  const ChangePath path = v.path = change_folds(plan, want_delta) ? kChangeFolded : kChangeFused;
  const std::vector<SosPar>& pars = v.tables.pars;
  const int unit = plan->d_mel_tc ? 128 : plan->TF;  // K1 work unit: a 128-frame block or a TF-frame tile
  v.T_k1.assign((size_t)n_clips, 0);
  v.pidx.assign((size_t)n_clips, int2{0, 0});
  v.first_unit.assign((size_t)n_clips + 1, 0);
  // the longest batched clip has the largest chunk of either cascade and needs the most shared memory: its tables
  // and size go to the launches
  int t_big = 0;
  for (int64_t i = 0; i < n_clips; ++i) {
    const int T = v.T_all[i];
    int a = -1, b = -1;
    ChangeRoute r{kChangeUnfused, kMfccFp32, 0};
    if (!plan->generic) {  // K1's ragged walk does not take the generic n_fft path
      a = v.tables.index(0, sa, T);
      b = out_iir ? v.tables.index(1, so, T) : a;
      r = change_route(plan, want_delta, first, rows, T, out_iir, a >= 0 ? &pars[a] : nullptr,
                       b >= 0 ? &pars[b] : nullptr, 1);
    }
    const bool ok = r.path == path && (path == kChangeFolded || r.k3 == kMfccFp32);
    const uint64_t units = v.first_unit[i] + (ok ? (uint64_t)(T + unit - 1) / unit : 0);
    if (units > 0x7fffffffULL) return fail(MMF_ERR_UNSUPPORTED, "variable-length batch of more than 2^31 K1 blocks");
    v.first_unit[i + 1] = (unsigned)units;
    if (!ok) {
      v.fallback.push_back(i);
      continue;
    }
    v.T_k1[i] = T;
    v.pidx[i] = int2{a, b};
    v.clips.push_back((int)i);
    if (T > t_big) {
      t_big = T;
      v.fsmem = r.smem;
      v.i1 = a;
      v.i2 = b;
    }
  }
  const int64_t nv = (int64_t)v.clips.size();
  if (!nv) v.tables.pars.clear();  // every clip takes the single-clip path: no launch reads the tables
  v.split_out = change_split_out(out_iir, nv);

  // workspace: descriptors, then the batched intermediates, then the single-clip region
  const size_t n = (size_t)n_clips;
  const int pitch = v.pitch;
  v.o_len = v.desc.put(v.len);
  v.o_tall = v.desc.put(v.T_all);
  v.o_tk1 = v.desc.put(v.T_k1);
  v.o_first = v.desc.put(v.first_unit);
  v.o_clips = v.desc.put(v.clips);
  v.o_pidx = v.desc.put(v.pidx);
  v.o_pars = v.desc.put(pars);
  size_t off = align_up(v.desc.size(), 256);
  v.o_logmel = (nv && !want_logmel) ? ws_take(off, n * c.n_mels * pitch * 4) : 0;
  v.o_clipmax = ws_take(off, n * 4);
  v.o_mfcc = (nv && path == kChangeFused && !want_mfcc) ? ws_take(off, n * c.n_mfcc * pitch * 4) : 0;
  v.o_raw = v.split_out ? ws_take(off, n * pitch * 8) : 0;
  v.o_single = off;
  size_t single_bytes = 0;
  for (int64_t i : v.fallback) {
    const size_t Ti = (size_t)v.T_all[i];
    size_t b = change_ws_bytes(plan, 1, (int64_t)Ti, true, true, rows) + align_up(Ti * 8, 256);
    if (want_logmel) b += align_up((size_t)c.n_mels * Ti * 4, 256);
    if (want_mfcc) b += align_up((size_t)c.n_mfcc * Ti * 4, 256);
    if (want_delta) b += align_up((size_t)c.n_mfcc * Ti * 4, 256);
    single_bytes = std::max(single_bytes, b);
  }
  v.bytes = v.o_single + single_bytes;
  return MMF_OK;
}

// Device half: runs the batch routed by v on `st`, carving from `base` (v.bytes).  `dd`: v.desc already on the device
// (null: uploaded to `base` here, a copy that waits for the stream).  Clip i is the v.len[i] samples at
// pcm_dev + i * clip_stride; the outputs given must be the ones v was routed for.
static int change_varlen_run(mmf_plan* plan, const ChangeVarlen& v, unsigned char* base, const unsigned char* dd,
                             const float* pcm_dev, int64_t clip_stride, const mmf_change_params* prm, double* tot_dev,
                             float* logmel_dev, float* mfcc_dev, float* delta_dev, cudaStream_t st) {
  const mmf_config& c = plan->cfg;
  const int64_t n_clips = v.n_clips;
  const size_t n = (size_t)n_clips;
  const int pitch = v.pitch, first = v.first, rows = v.rows;
  const int64_t nv = (int64_t)v.clips.size();
  int rc;
  if (!dd) {
    MMF_CUDA(cudaMemcpyAsync(base, v.desc.bytes.data(), v.desc.size(), cudaMemcpyHostToDevice, st));
    dd = base;
  }
  const int* d_tall = (const int*)(dd + v.o_tall);
  const int* d_tk1 = (const int*)(dd + v.o_tk1);

  // ---- the batched clips: one launch per stage
  if (nv) {
    const int64_t n_max = *std::max_element(v.len.begin(), v.len.end());
    const Varlen vl{(const long*)(dd + v.o_len), d_tk1, (const unsigned*)(dd + v.o_first), (long)v.first_unit[n],
                    pitch};
    float* logmel = logmel_dev ? logmel_dev : (float*)(base + v.o_logmel);
    int* clipmax = (int*)(base + v.o_clipmax);
    if ((rc = run_stft(plan, pcm_dev, n_clips, n_max, clip_stride, nullptr, logmel, clipmax, st, &vl))) return rc;
    const FusedVarlen fvl{(const int*)(dd + v.o_clips), d_tall, (const SosPar*)(dd + v.o_pars),
                          (const int2*)(dd + v.o_pidx)};
    const int clamp = logmel_dev ? 1 : 0;
    double* raw = v.split_out ? (double*)(base + v.o_raw) : nullptr;
    const SosPar& pa = v.tables.pars[v.i1];
    const SosPar& po = v.tables.pars[v.i2];
    const bool folded = v.path == kChangeFolded;
    const FusedMfccArgs lm{plan->d_dct, plan->nc_pad, logmel, clipmax, c.n_mels, c.top_db, mfcc_dev, delta_dev, clamp};
    float* mfcc = nullptr;
    if (!folded) {
      mfcc = mfcc_dev ? mfcc_dev : (float*)(base + v.o_mfcc);
      if ((rc = mfcc_run(plan, kMfccFp32, logmel, clipmax, n_clips, pitch, mfcc, delta_dev, clamp, st, d_tk1)))
        return rc;
    }
    cudaError_t e = change_fused_launch(mfcc, nv, c.n_mfcc, first, rows, pitch, prm->diff_method, pa, po,
                                        v.split_out ? 1 : prm->out_kind, v.split_out ? raw : tot_dev, v.fsmem,
                                        folded ? &lm : nullptr, st, &fvl);
    if (e == cudaSuccess && v.split_out) e = sosfiltfilt_par_varlen_launch(raw, 0, nv, pitch, po, fvl, tot_dev, st);
    if (e != cudaSuccess) return cuda_fail(e, "change_fused_kernel (variable-length) launch");
  }

  // ---- the other clips: the single-clip path, copied into their padded rows
  for (int64_t i : v.fallback) {
    const size_t Ti = (size_t)v.T_all[i];
    unsigned char* cur = base + v.o_single + change_ws_bytes(plan, 1, (int64_t)Ti, true, true, rows);
    double* tot1 = (double*)carve(cur, Ti * 8);
    float* lm1 = logmel_dev ? (float*)carve(cur, (size_t)c.n_mels * Ti * 4) : nullptr;
    float* mf1 = mfcc_dev ? (float*)carve(cur, (size_t)c.n_mfcc * Ti * 4) : nullptr;
    float* dl1 = delta_dev ? (float*)carve(cur, (size_t)c.n_mfcc * Ti * 4) : nullptr;
    if ((rc = run_change(plan, base + v.o_single, pcm_dev + (size_t)i * clip_stride, 1, v.len[i], v.len[i], prm, tot1,
                         lm1, mf1, dl1, st)))
      return rc;
    MMF_CUDA(cudaMemcpyAsync(tot_dev + (size_t)i * pitch, tot1, Ti * 8, cudaMemcpyDeviceToDevice, st));
    auto rows_to = [&](float* dst, const float* src, int r) {
      return cudaMemcpy2DAsync(dst + (size_t)i * r * pitch, (size_t)pitch * 4, src, Ti * 4, Ti * 4, r,
                               cudaMemcpyDeviceToDevice, st);
    };
    if (lm1) MMF_CUDA(rows_to(logmel_dev, lm1, c.n_mels));
    if (mf1) MMF_CUDA(rows_to(mfcc_dev, mf1, c.n_mfcc));
    if (dl1) MMF_CUDA(rows_to(delta_dev, dl1, c.n_mfcc));
  }
  cudaError_t e = varlen_tails_launch((long)n_clips, d_tall, pitch, tot_dev, logmel_dev, c.n_mels, mfcc_dev, delta_dev,
                                      c.n_mfcc, st);
  if (e != cudaSuccess) return cuda_fail(e, "varlen_tails_kernel launch");
  return MMF_OK;
}

}  // namespace mmf

extern "C" {

// Variable-length batch.  Each clip takes the route its own mmf_mfcc_change call would take -- which is what makes
// its outputs bit-identical to that call: K1 is a decision of the configuration alone, the post-MFCC route
// (change_route) depends on the clip's T.  Clips on the batch's route run in one launch per stage for the whole batch,
// each with the chunk tables (SosPar) of its own length; any other clip runs the single-clip path in workspace and is
// copied into its padded rows.
int mmf_mfcc_change_varlen(mmf_plan* plan, const float* pcm_dev, int64_t n_clips, const int64_t* n_samples_host,
                           int64_t clip_stride, const mmf_change_params* prm, double* tot_dev, float* logmel_dev,
                           float* mfcc_dev, float* delta_dev, void* stream) {
  using namespace mmf;
  // the lengths first: these checks need neither a plan nor a device
  if (!n_samples_host) return fail(MMF_ERR_INVALID, "n_samples_host is NULL");
  if (n_clips < 1) return fail(MMF_ERR_INVALID, "n_clips must be positive");
  if (n_clips > 0x7fffffff) return fail(MMF_ERR_UNSUPPORTED, "more than 2^31 - 1 clips");
  for (int64_t i = 0; i < n_clips; ++i) {
    const int64_t n = n_samples_host[i];
    if (n < 1 || n > clip_stride) {
      char buf[160];
      std::snprintf(buf, sizeof(buf), "clip %lld: n_samples %lld must be in [1, clip_stride = %lld]", (long long)i,
                    (long long)n, (long long)clip_stride);
      return fail(MMF_ERR_INVALID, buf);
    }
  }
  if (!plan || !pcm_dev || !prm || !tot_dev) return fail(MMF_ERR_INVALID, "NULL argument");
  ChangeVarlen v;
  int rc = change_varlen_route(plan, n_clips, n_samples_host, prm, logmel_dev != nullptr, mfcc_dev != nullptr,
                               delta_dev != nullptr, 0, v);
  if (rc) return rc;
  MMF_CUDA(cudaSetDevice(plan->cfg.device));
  if ((rc = ensure_ws(plan, (64 << 10) + v.bytes))) return rc;
  return change_varlen_run(plan, v, (unsigned char*)plan->ws + (64 << 10), nullptr, pcm_dev, clip_stride, prm, tot_dev,
                           logmel_dev, mfcc_dev, delta_dev, (cudaStream_t)stream);
}

}  // extern "C"

namespace mmf {

// Chunk budget of the host-buffer calls, in bytes of float32 PCM on the device, from a sweep on B200 (bench e2e legs,
// 1024 x 10 s clips): float32 host input 8 / 16 / 24 / 32 / 48 / 96 MB -> 0.68 / 0.81 / 0.82 / 0.82 / 0.81 / 0.80 M
// audio-s/s (small chunks pay launch + copy set-up, large ones a longer unoverlapped head and tail); int16 host input
// moves half the bytes per clip and keeps gaining up to 96 MB (0.94 / 1.16 / 1.25 / 1.34 / 1.37 / 1.44 M)
constexpr size_t kHostChunkF32 = 32u << 20, kHostChunkI16 = 96u << 20;
// Scratch of one sub-batch of a ragged Hilbert envelope (two M-point float64 work buffers per clip, the chirp and the
// transformed chirp filter per distinct length, the twiddles): a batch over it runs as several sub-batches of the
// same few launches, a clip over it alone.  At 2 GB a sub-batch holds about 120 clips of 10 s at 16 kHz (M = 2^19),
// some 15 000 CTAs per pass-group launch.
constexpr size_t kHilbertScratch = 2ull << 30;

// Runs `body`, which queues work on both plan streams, then drains both streams whatever it returned: queued copies
// target caller-owned host buffers.  The body's error comes first.
template <typename Body>
static int run_and_drain(mmf_plan* plan, Body&& body) {
  const int rc = body();
  const cudaError_t e0 = cudaStreamSynchronize(plan->streams[0]);
  const cudaError_t e1 = cudaStreamSynchronize(plan->streams[1]);
  if (rc) return rc;
  if (e0 != cudaSuccess) return cuda_fail(e0, "host path, stream 0");
  if (e1 != cudaSuccess) return cuda_fail(e1, "host path, stream 1");
  return MMF_OK;
}

}  // namespace mmf

// pcm_host: float32 samples, or (pcm16 != 0) int16 samples converted on the device
static int features_host_impl(mmf_plan* plan, const void* pcm_host_v, int pcm16, int64_t n_clips, int64_t n_samples,
                              int64_t clip_stride, const mmf_change_params* prm, const mmf_modspec_params* mod,
                              double* tot_host, float* mfcc_host, float* delta_host, float* mag_host,
                              float* band_host) {
  const float* pcm_host = (const float*)pcm_host_v;
  const int16_t* pcm_host16 = (const int16_t*)pcm_host_v;
  if (!plan || !pcm_host_v || !prm || !tot_host) return fail(MMF_ERR_INVALID, "NULL argument");
  if (n_clips < 1 || n_samples < 1) return fail(MMF_ERR_INVALID, "n_clips and n_samples must be positive");
  if ((mag_host || band_host) && !mod) return fail(MMF_ERR_INVALID, "modulation outputs requested without parameters");
  MMF_CUDA(cudaSetDevice(plan->cfg.device));
  const mmf_config& c = plan->cfg;
  const int64_t T = mmf_num_frames(n_samples, c.n_fft, c.hop_length);
  if (T < 1) return fail(MMF_ERR_INVALID, "input too short for one frame");
  const int rows = std::max(1, c.n_mfcc - (prm->remove_first ? 1 : 0));
  const bool want_mod = mod && (mag_host || band_host) && mod->win > 0;
  int64_t n_win = 0;
  int nbins = 0;
  if (want_mod) {
    const int rc = validate_modspec(mod->win, mod->hop, mod->nfft, mod->n_bands, mod->band_lo, mod->band_hi,
                                    band_host != nullptr);
    if (rc) return rc;
    n_win = T >= mod->win ? 1 + (T - mod->win) / mod->hop : 0;
    nbins = mod->nfft / 2 + 1;
  }
  const bool need_mfcc_dev = mfcc_host || want_mod;
  // chunk the batch so that H2D of chunk i+1 overlaps compute of chunk i (two streams, two slots)
  const size_t clip_bytes = (size_t)n_samples * 4;
  const size_t chunk_bytes = pcm16 ? kHostChunkI16 : kHostChunkF32;
  int64_t chunk = std::max<int64_t>(1, (int64_t)(chunk_bytes / clip_bytes));
  chunk = std::min<int64_t>(chunk, n_clips);
  const size_t pcm_slot = align_up((size_t)chunk * n_samples * 4, 256);
  const size_t tot_slot = align_up((size_t)chunk * T * 8, 256);
  const size_t mfcc_slot = need_mfcc_dev ? align_up((size_t)chunk * c.n_mfcc * T * 4, 256) : 0;
  const size_t delta_slot = delta_host ? align_up((size_t)chunk * c.n_mfcc * T * 4, 256) : 0;
  const size_t mag_slot = (want_mod && mag_host) ? align_up((size_t)chunk * c.n_mfcc * n_win * nbins * 4, 256) : 0;
  const size_t band_slot = (want_mod && band_host) ? align_up((size_t)chunk * n_win * mod->n_bands * 4 + 4, 256) : 0;
  const size_t change_slot = change_ws_bytes(plan, chunk, T, true, !need_mfcc_dev, rows);
  const size_t raw_slot = pcm16 ? align_up((size_t)chunk * n_samples * 2, 256) : 0;  // int16 staging
  const size_t slot = pcm_slot + raw_slot + tot_slot + mfcc_slot + delta_slot + mag_slot + band_slot + change_slot;
  int rc = ensure_host_ws(plan, (64 << 10) + 2 * slot);
  if (rc) return rc;
  // the modulation tables are (re)built with a device-wide synchronisation: do it before any copy is queued
  if (want_mod && n_win > 0 &&
      (rc = ensure_mod_tables(plan, mod->win, mod->nfft, mod->band_lo, mod->band_hi, band_host ? mod->n_bands : 0)))
    return rc;
  return run_and_drain(plan, [&]() -> int {
  int64_t done = 0;
  for (int i = 0; done < n_clips; ++i, done += chunk) {
    const int s = i & 1;
    const int64_t nc = std::min<int64_t>(chunk, n_clips - done);
    cudaStream_t st = plan->streams[s];
    unsigned char* cur = (unsigned char*)plan->host_ws + (64 << 10) + (size_t)s * slot;  // (unused: size 0)
    float* d_pcm = (float*)carve(cur, pcm_slot);
    int16_t* d_raw = (int16_t*)carve(cur, raw_slot);
    double* d_tot = (double*)carve(cur, tot_slot);
    float* d_mfcc = need_mfcc_dev ? (float*)carve(cur, mfcc_slot) : nullptr;
    float* d_delta = delta_host ? (float*)carve(cur, delta_slot) : nullptr;
    float* d_mag = mag_slot ? (float*)carve(cur, mag_slot) : nullptr;
    float* d_band = band_slot ? (float*)carve(cur, band_slot) : nullptr;
    // stream order serialises reuse of slot s (chunk i-2 ran on the same stream)
    if (pcm16) {
      if (clip_stride == n_samples) {
        MMF_CUDA(cudaMemcpyAsync(d_raw, pcm_host16 + (size_t)done * clip_stride, (size_t)nc * n_samples * 2,
                                 cudaMemcpyHostToDevice, st));
      } else {
        MMF_CUDA(cudaMemcpy2DAsync(d_raw, (size_t)n_samples * 2, pcm_host16 + (size_t)done * clip_stride,
                                   (size_t)clip_stride * 2, (size_t)n_samples * 2, (size_t)nc, cudaMemcpyHostToDevice,
                                   st));
      }
      cudaError_t ce = pcm16_to_f32_launch(d_raw, (long)nc * n_samples, d_pcm, st);
      if (ce != cudaSuccess) return cuda_fail(ce, "pcm16_to_f32_kernel launch");
    } else if (clip_stride == n_samples) {
      MMF_CUDA(cudaMemcpyAsync(d_pcm, pcm_host + (size_t)done * clip_stride, (size_t)nc * n_samples * 4,
                               cudaMemcpyHostToDevice, st));
    } else {
      MMF_CUDA(cudaMemcpy2DAsync(d_pcm, (size_t)n_samples * 4, pcm_host + (size_t)done * clip_stride,
                                 (size_t)clip_stride * 4, (size_t)n_samples * 4, (size_t)nc, cudaMemcpyHostToDevice,
                                 st));
    }
    // run_change carves its own scratch after a 64 KB constants area
    rc = run_change(plan, cur - (64 << 10), d_pcm, nc, n_samples, n_samples, prm, d_tot, nullptr, d_mfcc, d_delta, st);
    if (rc) return rc;
    if (want_mod && n_win > 0) {
      if ((rc = run_modspec(plan, d_mfcc, nc, c.n_mfcc, T, mod->win, mod->hop, mod->nfft, d_mag, d_band, mod->band_lo,
                            mod->band_hi, mod->n_bands, st)))
        return rc;
    }
    MMF_CUDA(cudaMemcpyAsync(tot_host + (size_t)done * T, d_tot, (size_t)nc * T * 8, cudaMemcpyDeviceToHost, st));
    if (mfcc_host)
      MMF_CUDA(cudaMemcpyAsync(mfcc_host + (size_t)done * c.n_mfcc * T, d_mfcc, (size_t)nc * c.n_mfcc * T * 4,
                               cudaMemcpyDeviceToHost, st));
    if (delta_host)
      MMF_CUDA(cudaMemcpyAsync(delta_host + (size_t)done * c.n_mfcc * T, d_delta, (size_t)nc * c.n_mfcc * T * 4,
                               cudaMemcpyDeviceToHost, st));
    if (d_mag && n_win > 0)
      MMF_CUDA(cudaMemcpyAsync(mag_host + (size_t)done * c.n_mfcc * n_win * nbins, d_mag,
                               (size_t)nc * c.n_mfcc * n_win * nbins * 4, cudaMemcpyDeviceToHost, st));
    if (d_band && n_win > 0)
      MMF_CUDA(cudaMemcpyAsync(band_host + (size_t)done * n_win * mod->n_bands, d_band,
                               (size_t)nc * n_win * mod->n_bands * 4, cudaMemcpyDeviceToHost, st));
  }
  return MMF_OK;
  });
}

namespace mmf {

// offsets[n_clips + 1] of a packed batch: non-decreasing from offsets[0] >= 0, every clip at least one sample (no plan
// or device needed)
static int validate_offsets(int64_t n_clips, const int64_t* offsets) {
  if (!offsets) return fail(MMF_ERR_INVALID, "offsets is NULL");
  if (n_clips < 1) return fail(MMF_ERR_INVALID, "n_clips must be positive");
  if (n_clips > 0x7fffffff) return fail(MMF_ERR_UNSUPPORTED, "more than 2^31 - 1 clips");
  if (offsets[0] < 0) return fail(MMF_ERR_INVALID, "clip 0: offsets[0] must be >= 0");
  for (int64_t i = 0; i < n_clips; ++i)
    if (offsets[i + 1] <= offsets[i]) {
      char buf[192];
      std::snprintf(buf, sizeof(buf), "clip %lld: offsets[%lld] = %lld, offsets[%lld] = %lld: every clip needs at least "
                    "one sample, in buffer order", (long long)i, (long long)i, (long long)offsets[i],
                    (long long)(i + 1), (long long)offsets[i + 1]);
      return fail(MMF_ERR_INVALID, buf);
    }
  return MMF_OK;
}

// Resampling descriptors of a packed batch (mmf_features_host_varlen_resampled, mmf_resample_varlen), after the
// offsets passed validate_offsets; no plan or device needed.  Taps are checked only for the clips that read them;
// *n_taps (0 on entry) becomes n_h when some clip does.
static int validate_resample(int64_t n_clips, const int64_t* offsets, const mmf_resample_clip* rs, const float* h,
                             int64_t n_h, int64_t* n_taps) {
  if (!rs) return fail(MMF_ERR_INVALID, "rs_host is NULL");
  for (int64_t i = 0; i < n_clips; ++i) {
    const mmf_resample_clip& r = rs[i];
    const int64_t len = offsets[i + 1] - offsets[i];
    char buf[256];
    auto bad = [&](const char* what) {
      std::snprintf(buf, sizeof(buf), "clip %lld: %s (up %d, down %d, tap0 %lld, len_h %d, n_pre_remove %lld, n_out "
                    "%lld, %lld samples, %lld taps)", (long long)i, what, r.up, r.down, (long long)r.tap0, r.len_h,
                    (long long)r.n_pre_remove, (long long)r.n_out, (long long)len, (long long)n_h);
      return fail(MMF_ERR_INVALID, buf);
    };
    if (r.up < 1 || r.down < 1) return bad("up and down must be >= 1");
    const bool copy = r.up == 1 && r.down == 1;
    const __int128 num = (__int128)len * r.up;
    if (r.n_out != (int64_t)((num + r.down - 1) / r.down))
      return bad(copy ? "a clip at the plan's rate needs n_out = its length" : "n_out must be ceil(len * up / down)");
    if (copy) continue;
    *n_taps = n_h;
    if (r.len_h < 1 || r.len_h > (1 << 22)) return bad("len_h must be in [1, 2^22]");
    if (!h || r.tap0 < 0 || r.tap0 > n_h - r.len_h) return bad("taps [tap0, tap0 + len_h) must lie in the tap table");
    if (r.n_pre_remove < 0) return bad("n_pre_remove must be >= 0");
  }
  return MMF_OK;
}

// Descriptors of clips [c0, c1) of a packed batch for resample_rows_launch, appended to `desc`.  Sources count from
// `base`; rs == NULL: every clip at the plan's rate.
static RaggedParts resample_desc(int64_t c0, int64_t c1, const int64_t* offsets, int64_t base,
                                 const mmf_resample_clip* rs, DescBlob& desc) {
  const int64_t nc = c1 - c0;
  std::vector<RsClip> cl((size_t)nc);
  std::vector<unsigned> first((size_t)nc + 1);
  int64_t items = 0;
  for (int64_t k = 0; k < nc; ++k) {
    const int64_t i = c0 + k, len = offsets[i + 1] - offsets[i];
    const long src = (long)(offsets[i] - base);
    if (!rs || (rs[i].up == 1 && rs[i].down == 1))
      cl[k] = RsClip{src, (long)len, 0, (long)len, 0, 0, 0, 0, 1};
    else
      cl[k] = RsClip{src, (long)len, (long)rs[i].n_pre_remove, (long)rs[i].n_out, (long)rs[i].tap0, rs[i].up,
                     rs[i].down, rs[i].len_h, 0};
    first[k] = (unsigned)items;
    items += (cl[k].n_out + kRsOut - 1) / kRsOut;
    if (items > 0x7fffffffLL) return RaggedParts{0, 0, -1};
  }
  first[nc] = (unsigned)items;
  return RaggedParts{desc.put(cl), desc.put(first), items};
}

// RMS-envelope geometry of a packed batch (mmf_amp_varlen_sizes, calc.py:326-331), after the offsets passed
// validate_offsets: amp_off[n_clips + 1], the prefix sums of each clip's frame count (no plan or device needed)
static int amp_sizes(int64_t n_clips, const int64_t* offsets, const int32_t* geom, int center, int64_t* amp_off) {
  if (!geom) return fail(MMF_ERR_INVALID, "geom_host is NULL");
  amp_off[0] = 0;
  for (int64_t i = 0; i < n_clips; ++i) {
    const int fl = geom[2 * i], hop = geom[2 * i + 1];
    const int64_t len = offsets[i + 1] - offsets[i];
    char buf[160];
    if (fl < 1 || hop < 1) {
      std::snprintf(buf, sizeof(buf), "clip %lld: frame_length (%d) and hop (%d) must be >= 1", (long long)i, fl, hop);
      return fail(MMF_ERR_INVALID, buf);
    }
    const int64_t padded = len + (center ? 2 * (int64_t)(fl / 2) : 0);
    if (padded < fl) {
      std::snprintf(buf, sizeof(buf), "clip %lld: Input is too short (n=%lld) for frame_length=%d", (long long)i,
                    (long long)len, fl);
      return fail(MMF_ERR_TOO_SHORT, buf);
    }
    amp_off[i + 1] = amp_off[i] + 1 + (padded - fl) / hop;
  }
  return MMF_OK;
}

// Envelope geometry of a packed batch (mmf_env_varlen_sizes) after the offsets passed validate_offsets: RMS as
// amp_sizes; Hilbert one output per sample, at most 2^26 samples per clip
static int env_sizes(int64_t n_clips, const int64_t* offsets, const mmf_env_params* env, const int32_t* geom,
                     int64_t* amp_off) {
  char buf[160];
  if (env->method == MMF_ENV_RMS) return amp_sizes(n_clips, offsets, geom, env->center, amp_off);
  if (env->method != MMF_ENV_HILBERT) {
    std::snprintf(buf, sizeof(buf), "unknown envelope method %d (MMF_ENV_RMS 0, MMF_ENV_HILBERT 1)", env->method);
    return fail(MMF_ERR_INVALID, buf);
  }
  amp_off[0] = 0;
  for (int64_t i = 0; i < n_clips; ++i) {
    const int64_t len = offsets[i + 1] - offsets[i];
    if (len > (1LL << 26)) {
      std::snprintf(buf, sizeof(buf), "clip %lld: %lld samples; the Hilbert envelope takes at most 2^26",
                    (long long)i, (long long)len);
      return fail(MMF_ERR_UNSUPPORTED, buf);
    }
    amp_off[i + 1] = amp_off[i] + len;
  }
  return MMF_OK;
}

// The Hilbert route of a batch: clips of at most kHilDirectMax samples one by one through the direct convolution
// (direct: n, src, out of each), the others in sub-batches of one hilbert_varlen_launch each
struct HilSub {
  size_t o_tab = 0, o_clip = 0, o_tab_first = 0, o_clip_first = 0, o_chirp_first = 0;  // in the route's DescBlob
  HilBatch b{};        // counts, groups and twiddle offset; the pointers are set at run time
  size_t scratch = 0;  // bytes of the sub-batch's scratch
};
struct HilbertVarlen {
  std::vector<HilSub> subs;
  std::vector<HilRow> direct;
};

static int hil_log2(long n) {
  int m = 0;
  while ((1L << m) < 2 * n - 1) ++m;
  return m;
}

// one sub-batch of the clips `rows` (n, src, out set): the tables of each distinct n, shared by its clips, the work
// buffers and the twiddles of the largest M in one scratch allocation (double2 offsets, 256-byte aligned regions);
// rows ordered three-group rows first
static void hilbert_sub(std::vector<HilRow> rows, HilbertVarlen& h, DescBlob& desc) {
  auto region = [](long& end, long elems) {
    const long o = end;
    end += (elems + 15) & ~15L;
    return o;
  };
  int mw = 0;
  for (const HilRow& r : rows) mw = std::max(mw, hil_log2(r.n));
  long end = 0;
  const long w = region(end, 1L << (mw - 1));
  std::vector<HilRow> tab;
  for (size_t k = 0; k < rows.size(); ++k) {
    HilRow& r = rows[k];
    r.m = hil_log2(r.n);
    r.G = hilbert_groups(r.m, r.L);
    r.inv_env = 1.0 / ((double)(1L << r.m) * (double)r.n);
    int t = -1;
    for (size_t q = 0; q < tab.size() && t < 0; ++q)
      if (tab[q].n == r.n) t = (int)q;
    if (t < 0) {
      t = (int)tab.size();
      HilRow tr = r;
      tr.c = region(end, r.n);
      tr.bf = tr.buf0 = region(end, 1L << r.m);
      tab.push_back(tr);
    }
    r.c = tab[t].c;
    r.bf = tab[t].bf;
    r.buf0 = region(end, 1L << r.m);
    r.buf1 = region(end, 1L << r.m);
    if (tab[t].buf1 == 0) tab[t].buf1 = r.buf0;  // the chirp filter's other buffer: its first clip's (offset 0 is w)
  }
  HilSub sb;
  HilBatch& b = sb.b;
  b.w = w;
  b.mw = mw;
  b.G = 2;
  auto order = [&](std::vector<HilRow>& v, long& n3, long& items, long& items3, size_t& o_rows, size_t& o_first) {
    std::stable_partition(v.begin(), v.end(), [](const HilRow& r) { return r.G == 3; });
    std::vector<unsigned> first(v.size() + 1, 0);
    n3 = 0;
    for (size_t k = 0; k < v.size(); ++k) {
      first[k + 1] = first[k] + (unsigned)hilbert_items(v[k].m);
      if (v[k].G == 3) n3 = (long)k + 1, b.G = 3;
    }
    items = first[v.size()];
    items3 = first[n3];
    o_rows = desc.put(v);
    o_first = desc.put(first);
  };
  b.n_tab = (long)tab.size();
  b.n_clip = (long)rows.size();
  order(tab, b.n_tab3, b.tab_items, b.tab_items3, sb.o_tab, sb.o_tab_first);
  order(rows, b.n_clip3, b.clip_items, b.clip_items3, sb.o_clip, sb.o_clip_first);
  std::vector<unsigned> chirp(tab.size() + 1, 0);
  for (size_t q = 0; q < tab.size(); ++q) chirp[q + 1] = chirp[q] + (unsigned)((tab[q].n + 255) / 256);
  b.chirp_items = chirp[tab.size()];
  sb.o_chirp_first = desc.put(chirp);
  sb.scratch = (size_t)end * 16;
  h.subs.push_back(sb);
}

// clips k < n.size(): n[k] samples at x + src[k], envelope at amp + out[k].  Sub-batches: maximal runs of the FFT
// clips whose scratch stays within kHilbertScratch
static void hilbert_route(const std::vector<long>& src, const std::vector<long>& n, const std::vector<long>& out,
                          HilbertVarlen& h, DescBlob& desc) {
  std::vector<HilRow> cur;
  std::vector<long> lens;
  size_t bytes = 0;
  int mw = 0;
  for (size_t k = 0; k < n.size(); ++k) {
    HilRow r{};
    r.n = n[k];
    r.src = src[k];
    r.out = out[k];
    if (n[k] <= kHilDirectMax) {
      h.direct.push_back(r);
      continue;
    }
    const int m = hil_log2(n[k]);
    const size_t M16 = ((size_t)16 << m) + 256, tables = M16 + (size_t)n[k] * 16 + 256;
    bool seen = std::find(lens.begin(), lens.end(), n[k]) != lens.end();
    if (!cur.empty() && bytes + 2 * M16 + (seen ? 0 : tables) + ((size_t)8 << std::max(mw, m)) > kHilbertScratch) {
      hilbert_sub(std::move(cur), h, desc);
      cur.clear();
      lens.clear();
      bytes = 0;
      mw = 0;
      seen = false;
    }
    cur.push_back(r);
    if (!seen) lens.push_back(n[k]);
    bytes += 2 * M16 + (seen ? 0 : tables);
    mw = std::max(mw, m);
  }
  if (!cur.empty()) hilbert_sub(std::move(cur), h, desc);
}

// Device half: every sub-batch in stream-ordered scratch, then the direct clips, on `st`.  dd: the descriptors there
static int hilbert_run(const HilbertVarlen& h, const unsigned char* dd, const void* x, int pcm16, float* amp,
                       int sm_count, cudaStream_t st) {
  for (const HilSub& sb : h.subs) {
    HilBatch b = sb.b;
    b.tab = (const HilRow*)(dd + sb.o_tab);
    b.clip = (const HilRow*)(dd + sb.o_clip);
    b.tab_first = (const unsigned*)(dd + sb.o_tab_first);
    b.clip_first = (const unsigned*)(dd + sb.o_clip_first);
    b.chirp_first = (const unsigned*)(dd + sb.o_chirp_first);
    b.x = x;
    b.pcm16 = pcm16;
    b.amp = amp;
    MMF_CUDA(cudaMallocAsync((void**)&b.s, sb.scratch, st));
    const cudaError_t e = hilbert_varlen_launch(b, st);
    cudaFreeAsync(b.s, st);
    if (e != cudaSuccess) return cuda_fail(e, "hilbert_group_kernel launch");
  }
  for (const HilRow& r : h.direct) {
    const void* xr = pcm16 ? (const void*)((const int16_t*)x + r.src) : (const void*)((const float*)x + r.src);
    const cudaError_t e = hilbert_envelope_launch(xr, pcm16, 1, r.n, r.n, amp + r.out, r.n, sm_count, st);
    if (e != cudaSuccess) return cuda_fail(e, "hilbert_conv_kernel launch");
  }
  return MMF_OK;
}

// Host half of a ragged RMS envelope (mmf_rms_varlen, the envelope of the host bundle): the descriptors of the
// envelope launch and, with an output filter, each envelope's route -- that of its own mmf_sosfiltfilt call: the
// chunk-parallel kernel when it takes the envelope's length (all of them in one launch, each with the tables of its
// own chunk length), the single-row routes otherwise.
struct EnvelopeVarlen {
  int method = MMF_ENV_RMS;
  HilbertVarlen hil;              // the Hilbert envelope's launches (method MMF_ENV_HILBERT)
  int64_t n_clips = 0;
  std::vector<int64_t> off;       // envelope k: frames [off[k], off[k + 1]) of the output
  const SosArgs* filt = nullptr;  // the output filter (null: none)
  SosParSet tables;
  int amax = -1;                  // the widest tables: they size the batched filter's launch
  std::vector<int> par;           // envelopes on the chunk-parallel route
  std::vector<int64_t> single;    // the others
  DescBlob desc;
  RaggedParts rms;                                               // the envelope launch (RmsClip)
  size_t o_par = 0, o_T = 0, o_pidx = 0, o_off = 0, o_pars = 0;  // the batched filter (FusedVarlen)
};

// Routing of clips [c0, c1) of a packed batch whose amp_sizes are amp_off (host only).  Sources count from `base`,
// outputs from amp_off[c0].  Returns the number of envelope work items, -1 past 2^31 - 1.
static void filter_route(EnvelopeVarlen& v);
static int64_t envelope_route(int64_t c0, int64_t c1, const int64_t* offsets, int64_t base, const int32_t* geom,
                              int center, const int64_t* amp_off, const SosArgs* filt, EnvelopeVarlen& v) {
  const int64_t nc = c1 - c0;
  v.n_clips = nc;
  v.filt = filt;
  v.off.resize((size_t)nc + 1);
  std::vector<RmsClip> cl((size_t)nc);
  std::vector<unsigned> first((size_t)nc + 1);
  int64_t items = 0;
  for (int64_t k = 0; k < nc; ++k) {
    const int64_t i = c0 + k;
    const int fl = geom[2 * i], hop = geom[2 * i + 1];
    v.off[k] = amp_off[i] - amp_off[c0];
    cl[k] = RmsClip{(long)(offsets[i] - base), (long)(offsets[i + 1] - offsets[i]), (long)v.off[k],
                    (long)(amp_off[i + 1] - amp_off[i]), fl, hop, center ? fl / 2 : 0, rms_frames_per_item(fl, hop)};
    first[k] = (unsigned)items;
    items += (cl[k].T + cl[k].F - 1) / cl[k].F;
    if (items > 0x7fffffffLL) return -1;
  }
  first[nc] = (unsigned)items;
  v.off[nc] = amp_off[c1] - amp_off[c0];
  v.rms = RaggedParts{v.desc.put(cl), v.desc.put(first), items};
  filter_route(v);
  return items;
}

// Hilbert routing of clips [c0, c1) (host only): sources count from `base`, outputs from amp_off[c0]
static void hilbert_env_route(int64_t c0, int64_t c1, const int64_t* offsets, int64_t base, const int64_t* amp_off,
                              const SosArgs* filt, EnvelopeVarlen& v) {
  const int64_t nc = c1 - c0;
  v.method = MMF_ENV_HILBERT;
  v.n_clips = nc;
  v.filt = filt;
  v.off.resize((size_t)nc + 1);
  std::vector<long> src((size_t)nc), n((size_t)nc), out((size_t)nc);
  for (int64_t k = 0; k <= nc; ++k) v.off[k] = amp_off[c0 + k] - amp_off[c0];
  for (int64_t k = 0; k < nc; ++k) {
    src[k] = (long)(offsets[c0 + k] - base);
    n[k] = (long)(offsets[c0 + k + 1] - offsets[c0 + k]);
    out[k] = (long)v.off[k];
  }
  hilbert_route(src, n, out, v.hil, v.desc);
  filter_route(v);
}

// With an output filter, each envelope's route: that of its own mmf_sosfiltfilt call (see EnvelopeVarlen)
static void filter_route(EnvelopeVarlen& v) {
  if (!v.filt) return;
  const int64_t nc = v.n_clips;
  const SosArgs* filt = v.filt;
  std::vector<int> T((size_t)nc);
  std::vector<int2> pidx((size_t)nc, int2{0, 0});
  for (int64_t k = 0; k < nc; ++k) {
    const int64_t Tk = v.off[k + 1] - v.off[k];
    T[k] = (int)std::min<int64_t>(Tk, 0x7fffffff);
    const int idx = v.tables.index(0, *filt, (long)Tk);
    if (idx < 0) {
      v.single.push_back(k);
      continue;
    }
    if (v.amax < 0 || v.tables.pars[idx].CL > v.tables.pars[v.amax].CL) v.amax = idx;
    pidx[k] = int2{idx, idx};
    v.par.push_back((int)k);
  }
  v.o_par = v.desc.put(v.par);
  v.o_T = v.desc.put(T);
  v.o_pidx = v.desc.put(pidx);
  v.o_off = v.desc.put(v.off.data(), (size_t)nc);
  v.o_pars = v.desc.put(v.tables.pars);
}

// Device half: the envelope launch over x (float32, or int16 when pcm16) into amp and, with the output filter, the
// batched filter launch and the single-row filters into amp_filt, all on `st`.  dd: v.desc on the device.
static int envelope_run(const EnvelopeVarlen& v, const unsigned char* dd, const void* x, int pcm16, float* amp,
                        double* amp_filt, int sm_count, cudaStream_t st) {
  cudaError_t e;
  if (v.method == MMF_ENV_HILBERT) {
    if (const int rc = hilbert_run(v.hil, dd, x, pcm16, amp, sm_count, st)) return rc;
  } else {
    e = rms_varlen_launch(x, pcm16, (const RmsClip*)(dd + v.rms.clips), (const unsigned*)(dd + v.rms.first),
                          (long)v.n_clips, (long)v.rms.items, amp, st);
    if (e != cudaSuccess) return cuda_fail(e, "rms_varlen_kernel launch");
  }
  if (amp_filt && !v.par.empty()) {
    const FusedVarlen fvl{(const int*)(dd + v.o_par), (const int*)(dd + v.o_T), (const SosPar*)(dd + v.o_pars),
                          (const int2*)(dd + v.o_pidx), (const long*)(dd + v.o_off)};
    e = sosfiltfilt_par_varlen_launch(amp, 1, (long)v.par.size(), 0, v.tables.pars[v.amax], fvl, amp_filt, st);
    if (e != cudaSuccess) return cuda_fail(e, "sosfiltfilt_par_kernel (envelopes) launch");
  }
  for (int64_t k : v.single) {
    const int64_t a0 = v.off[k], Tk = v.off[k + 1] - v.off[k];
    e = sosfiltfilt_any(amp + a0, 1, 1, (long)Tk, (long)Tk, 1, 0, *v.filt, amp_filt + a0, (long)Tk, st);
    if (e != cudaSuccess) return cuda_fail(e, "sosfiltfilt (envelope)");
  }
  return MMF_OK;
}

// Uploads `desc` to stream-ordered scratch on `st` and runs launch(its device address) there; the scratch is freed in
// stream order after it.  (A pageable source: the copy is staged, so the host blob may go when this returns.)
template <typename Launch>
static int run_uploaded(mmf_plan* plan, const DescBlob& desc, cudaStream_t st, Launch&& launch) {
  MMF_CUDA(cudaSetDevice(plan->cfg.device));
  if (!desc.size()) return launch(nullptr);
  unsigned char* d = nullptr;
  MMF_CUDA(cudaMallocAsync((void**)&d, desc.size(), st));
  const cudaError_t e = cudaMemcpyAsync(d, desc.bytes.data(), desc.size(), cudaMemcpyHostToDevice, st);
  const int rc = e != cudaSuccess ? cuda_fail(e, "descriptor upload") : launch((const unsigned char*)d);
  cudaFreeAsync(d, st);
  return rc;
}

// ---- the 'fir' / 'sg' output filters over ragged rows (fir_varlen_launch, stencil_varlen_launch) ----

// The checks of a filter's kind and coefficients, which do not depend on the rows
static int filter_shape_check(const mmf_out_filter* f) {
  if (!f) return fail(MMF_ERR_INVALID, "output filter is NULL");
  if (f->kind == MMF_FILT_FIR) {
    if (f->n_taps < 1 || f->n_taps > 4096) return fail(MMF_ERR_UNSUPPORTED, "n_taps must be in [1, 4096]");
    if (!f->taps) return fail(MMF_ERR_INVALID, "taps is NULL");
    return MMF_OK;
  }
  if (f->kind != MMF_FILT_SG) return fail(MMF_ERR_INVALID, "unknown output filter kind " + std::to_string(f->kind));
  if (!f->coef) return fail(MMF_ERR_INVALID, "coef is NULL");
  if (f->half < 0 || f->n_edge < f->half || f->n_edge_in < 0) return fail(MMF_ERR_INVALID, "need n_edge >= half >= 0");
  if (f->n_edge > 0 && (!f->edge_l || !f->edge_r)) return fail(MMF_ERR_INVALID, "edge matrices are NULL");
  return MMF_OK;
}

// A row of T samples too short for f: the single calls' error, naming the row when clip >= 0
static int filter_row_check(const mmf_out_filter* f, int64_t T, int64_t clip) {
  if (f->kind == MMF_FILT_FIR) return T <= 3 * (int64_t)f->n_taps ? too_short(3 * f->n_taps, clip) : MMF_OK;
  if (T < f->n_edge_in || T < 2 * (int64_t)f->n_edge)
    return fail(MMF_ERR_TOO_SHORT, (clip < 0 ? "" : "clip " + std::to_string(clip) + ": ") +
                                       "input shorter than the stencil's edge window");
  return MMF_OK;
}

// A ragged output-filter launch, host half: the rows, their work lists and the coefficients, in desc.  The FIR's
// forward-pass scratch is packed row after row (work: its size in doubles).
struct FilterVarlen {
  int64_t n_rows = 0, work = 0;
  RaggedParts a, b;  // SG: a; FIR: a the forward pass, b the backward pass (the same rows)
  size_t taps = 0, coef = 0, el = 0, er = 0;
  DescBlob desc;
};

// rows i < n: T[i] samples at x_off[i], outputs at y_off[i]; the rows passed filter_row_check
static int filter_route(const mmf_out_filter* f, int64_t n, const int64_t* x_off, const int64_t* T,
                        const int64_t* y_off, FilterVarlen& v) {
  const bool fir = f->kind == MMF_FILT_FIR;
  const int64_t ext = fir ? 6 * (int64_t)f->n_taps : 0;
  std::vector<FiltRow> rows((size_t)n);
  std::vector<unsigned> fa((size_t)n + 1), fb((size_t)n + 1);
  int64_t ia = 0, ib = 0, w = 0;
  for (int64_t i = 0; i < n; ++i) {
    rows[i] = FiltRow{(long)x_off[i], (long)T[i], (long)y_off[i], (long)w};
    fa[i] = (unsigned)ia;
    fb[i] = (unsigned)ib;
    ia += (T[i] + ext + kFiltOut - 1) / kFiltOut;
    ib += (T[i] + kFiltOut - 1) / kFiltOut;
    w += T[i] + ext;
    if (ia > 0x7fffffffLL) return fail(MMF_ERR_UNSUPPORTED, "more than 2^31 - 1 work items");
  }
  fa[n] = (unsigned)ia;
  fb[n] = (unsigned)ib;
  v.n_rows = n;
  v.a = RaggedParts{v.desc.put(rows), v.desc.put(fa), ia};
  if (fir) {
    v.b = RaggedParts{v.a.clips, v.desc.put(fb), ib};
    v.taps = v.desc.put(f->taps, (size_t)f->n_taps);
    v.work = w;
  } else {
    v.coef = v.desc.put(f->coef, (size_t)(2 * f->half + 1));
    const size_t ne = (size_t)f->n_edge * f->n_edge_in;
    if (ne) {
      v.el = v.desc.put(f->edge_l, ne);
      v.er = v.desc.put(f->edge_r, ne);
    }
  }
  return MMF_OK;
}

// The device half on `st`: d, v.desc on the device; work: v.work doubles (FIR)
static int filter_run(const mmf_out_filter* f, const FilterVarlen& v, const unsigned char* d, const void* x,
                      int x_is_f32, double* y, double* work, cudaStream_t st) {
  const FiltRow* rows = (const FiltRow*)(d + v.a.clips);
  if (f->kind == MMF_FILT_FIR) {
    const cudaError_t e = fir_varlen_launch(x, x_is_f32, rows, (long)v.n_rows, (const unsigned*)(d + v.a.first),
                                            (long)v.a.items, (const unsigned*)(d + v.b.first), (long)v.b.items,
                                            (const double*)(d + v.taps), f->n_taps, work, y, st);
    return e == cudaSuccess ? MMF_OK : cuda_fail(e, "fir kernels launch");
  }
  const bool edges = (size_t)f->n_edge * f->n_edge_in > 0;
  const cudaError_t e = stencil_varlen_launch(x, x_is_f32, rows, (long)v.n_rows, (const unsigned*)(d + v.a.first),
                                              (long)v.a.items, (const double*)(d + v.coef), f->half,
                                              edges ? (const double*)(d + v.el) : nullptr,
                                              edges ? (const double*)(d + v.er) : nullptr, f->n_edge, f->n_edge_in,
                                              y, st);
  return e == cudaSuccess ? MMF_OK : cuda_fail(e, "stencil_varlen_kernel launch");
}

// One ragged filter launch on `st` with descriptors uploaded; work: caller's FIR scratch, else the stream-ordered pool
static int filter_uploaded(mmf_plan* plan, const mmf_out_filter* f, const FilterVarlen& v, const void* x,
                           int x_is_f32, double* y, double* work, cudaStream_t st) {
  return run_uploaded(plan, v.desc, st, [&](const unsigned char* d) {
    double* pool = nullptr;
    if (!work && v.work) MMF_CUDA(cudaMallocAsync((void**)&pool, (size_t)v.work * sizeof(double), st));
    const int rc = filter_run(f, v, d, x, x_is_f32, y, work ? work : pool, st);
    if (pool) cudaFreeAsync(pool, st);
    return rc;
  });
}

// One ragged envelope (RMS or Hilbert) on `st` over float32 x from the host descriptors of v (no output filter)
static int rms_run(mmf_plan* plan, const float* x, const EnvelopeVarlen& v, float* out, cudaStream_t st) {
  return run_uploaded(plan, v.desc, st, [&](const unsigned char* d) {
    return envelope_run(v, d, x, 0, out, nullptr, plan->sm_count, st);
  });
}

// One ragged resampling launch on `st`: the descriptors at p of `desc`, which takes the taps h[n_h]
static int resample_dev(mmf_plan* plan, const float* x_dev, DescBlob& desc, const RaggedParts& p, const float* h,
                        int64_t n_h, int64_t n_clips, float* y_dev, int64_t y_stride, cudaStream_t st) {
  const size_t o_h = desc.put(h, (size_t)n_h);
  return run_uploaded(plan, desc, st, [&](const unsigned char* d) {
    const cudaError_t e = resample_rows_launch(x_dev, 0, (const RsClip*)(d + p.clips), (const unsigned*)(d + p.first),
                                               (long)n_clips, (long)p.items, (const float*)(d + o_h), y_dev,
                                               (long)y_stride, st);
    return e == cudaSuccess ? MMF_OK : cuda_fail(e, "resample_rows_kernel launch");
  });
}

// frame_off / win_off of a packed batch (mmf_features_varlen_sizes); n_win_i = 0 without modulation windows
static void packed_sizes(int n_fft, int hop, int win, int mod_hop, int64_t n_clips, const int64_t* offsets,
                         int64_t* frame_off, int64_t* win_off) {
  frame_off[0] = win_off[0] = 0;
  for (int64_t i = 0; i < n_clips; ++i) {
    const int64_t T = mmf_num_frames(offsets[i + 1] - offsets[i], n_fft, hop);
    frame_off[i + 1] = frame_off[i] + T;
    win_off[i + 1] = win_off[i] + (win > 0 && T >= win ? 1 + (T - win) / mod_hop : 0);
  }
}

// A packed host-buffer call: the arguments of the packed entry points in their order, then what the host-only checks
// derive from them.  pcm: float32 samples, or (pcm16 != 0) int16 samples converted on the device.  resampled: clip i
// reaches the plan's rate as rs[i] says, with taps from h_taps[n_h]; otherwise every clip is at the plan's rate.
// env_prm: the envelope of each clip's native samples (RMS: frame geometry geom[2i], geom[2i + 1]; Hilbert: one
// output per sample), to amp and / or,
// through the output filter, amp_filt (NULL: none, and exactly the launches and copies of the call without it).
struct PackedBatch {
  const void* pcm;
  int pcm16;
  int64_t n_clips;
  const int64_t* offsets;
  const mmf_resample_clip* rs;
  const float* h_taps;
  int64_t n_h;
  const mmf_change_params* prm;
  const mmf_modspec_params* mod;
  const mmf_env_params* env_prm;
  const int32_t* geom;
  double* tot;
  float *mfcc, *delta, *mag, *band;
  float* amp = nullptr;
  double* amp_filt = nullptr;
  bool resampled = false;
  const mmf_out_filter* change_out = nullptr;  // the MFCC-change curve's 'fir' / 'sg' filter (NULL: none)
  size_t isz = pcm16 ? 2 : 4;  // bytes per sample as they cross PCIe
  // from the checks
  int64_t n_taps = 0;  // taps that go up with the descriptors: none unless some clip reads them
  bool want_mod = false, want_amp = false, need_mfcc_dev = false;
  int nb = 0, nbe = 0;  // modulation bins per window; band outputs actually written
  SosArgs amp_sos;      // the envelopes' output filter (amp_filt)
  // len: samples at the plan's rate (what the ragged path sees); T: frames.  F, Wo, A [n_clips + 1]: packed offsets
  // of frames, modulation windows and envelope frames
  std::vector<int64_t> len, T, F, Wo, A;
};

// Byte offsets of a chunk's buffers in its slot of the host-path workspace, in the order they are laid out
struct HostSlot {
  size_t h2d = 0, pcm = 0, tot = 0, mfcc = 0, delta = 0, mag = 0, band = 0;
  size_t ptot = 0, pmfcc = 0, pdelta = 0, pmag = 0, pband = 0, scratch = 0, amp = 0, amp_filt = 0, ctot = 0,
         cwork = 0, end = 0;
};

// per-clip row lengths (int) and packed offsets (long) of a compaction, in the call's descriptors
struct PackedRows {
  size_t cnt = 0, off = 0;
};

// One chunk of a packed host-buffer batch: a run of consecutive clips, its routed stages and its slot
struct HostChunk {
  // clips [c0, c1); stride: samples per staged row, the chunk's longest clip rounded up to 16 bytes for the TMA
  int64_t c0 = 0, c1 = 0, stride = 0;
  RaggedParts stage;       // the staging launch (resample_rows_launch)
  PackedRows frames, wins;  // compaction of the per-frame and the per-window outputs
  ChangeVarlen cv;
  ModspecVarlen mv;    // routed when the chunk has modulation windows (mv.W > 0)
  EnvelopeVarlen env;  // routed when the envelope is requested
  FilterVarlen fv;     // the change curve's output filter, over the padded [nc, pitch] rows (change_out only)
  size_t o_cv = 0, o_mv = 0, o_env = 0, o_fv = 0;  // cv.desc, mv.desc, env.desc and fv.desc in the call's descriptors
  HostSlot slot;
};

// Stage 1 (host only): the checks that precede routing, in the order the callers see them, and the packed sizes
static int packed_check(const mmf_plan* plan, PackedBatch& b) {
  const mmf_env_params* amp = b.env_prm;
  int rc = validate_offsets(b.n_clips, b.offsets);
  if (rc) return rc;
  if (b.resampled && (rc = validate_resample(b.n_clips, b.offsets, b.rs, b.h_taps, b.n_h, &b.n_taps))) return rc;
  if (!amp && (b.amp || b.amp_filt)) return fail(MMF_ERR_INVALID, "amplitude outputs requested without parameters");
  const size_t n = (size_t)b.n_clips;
  b.want_amp = amp && (b.amp || b.amp_filt);
  if (b.want_amp) {
    b.A.resize(n + 1);
    if ((rc = env_sizes(b.n_clips, b.offsets, amp, b.geom, b.A.data()))) return rc;
    if (b.amp_filt) {
      if (amp->out_n_sections < 1) return fail(MMF_ERR_INVALID, "amp_filt_host needs out_n_sections >= 1");
      if ((rc = fill_sos(amp->out_sos, amp->out_n_sections, &b.amp_sos))) return rc;
      for (size_t i = 0; i < n; ++i)
        if (b.A[i + 1] - b.A[i] <= b.amp_sos.padlen) return too_short(b.amp_sos.padlen, (int64_t)i);
    }
  }
  if (b.change_out) {
    if ((rc = filter_shape_check(b.change_out))) return rc;
    if (b.prm && b.prm->out_kind != 1)
      return fail(MMF_ERR_INVALID, "change_out needs prm->out_kind == 1 (the raw curve)");
  }
  if (!plan || !b.pcm || !b.prm || !b.tot) return fail(MMF_ERR_INVALID, "NULL argument");
  if ((b.mag || b.band) && !b.mod) return fail(MMF_ERR_INVALID, "modulation outputs requested without parameters");
  const mmf_modspec_params* mod = b.mod;
  b.want_mod = mod && (b.mag || b.band) && mod->win > 0;
  if (b.want_mod && (rc = validate_modspec(mod->win, mod->hop, mod->nfft, mod->n_bands, mod->band_lo, mod->band_hi,
                                           b.band != nullptr)))
    return rc;
  b.nb = b.want_mod ? mod->nfft / 2 + 1 : 0;
  b.nbe = b.want_mod && b.band ? mod->n_bands : 0;
  b.need_mfcc_dev = b.mfcc || b.want_mod;
  b.len = b.T = std::vector<int64_t>(n);
  b.F = b.Wo = std::vector<int64_t>(n + 1);
  std::vector<int64_t> out_off(n + 1, 0);
  for (size_t i = 0; i < n; ++i) {
    b.len[i] = b.rs ? b.rs[i].n_out : b.offsets[i + 1] - b.offsets[i];
    out_off[i + 1] = out_off[i] + b.len[i];
  }
  packed_sizes(plan->cfg.n_fft, plan->cfg.hop_length, b.want_mod ? mod->win : 0, b.want_mod ? mod->hop : 1, b.n_clips,
               out_off.data(), b.F.data(), b.Wo.data());
  for (size_t i = 0; i < n; ++i) b.T[i] = b.F[i + 1] - b.F[i];
  return MMF_OK;
}

// A chunk's routing, with every check in stage order, and its staging and compaction descriptors, appended to the
// call's
static int route_chunk(const mmf_plan* plan, const PackedBatch& b, HostChunk& h, DescBlob& desc) {
  const int64_t c0 = h.c0, c1 = h.c1, nc = c1 - c0;
  int rc = change_varlen_route(plan, nc, b.len.data() + c0, b.prm, false, b.need_mfcc_dev, b.delta != nullptr, c0,
                               h.cv);
  if (rc) return rc;
  int64_t W = 0;
  for (int64_t i = c0; i < c1; ++i) W = std::max(W, b.Wo[i + 1] - b.Wo[i]);
  if (W > 0x7fffffff) return fail(MMF_ERR_UNSUPPORTED, "more than 2^31 - 1 windows per clip");
  if (b.want_mod && W > 0 &&
      (rc = modspec_varlen_route((unsigned)plan->cfg.flags, b.T.data() + c0, nc, plan->cfg.n_mfcc, W, b.mod->win,
                                 b.mod->hop, b.mod->nfft, b.nbe, b.mag != nullptr, h.mv)))
    return rc;
  h.stage = resample_desc(c0, c1, b.offsets, b.offsets[c0], b.rs, desc);
  if (h.stage.items < 0) return fail(MMF_ERR_UNSUPPORTED, "a chunk of more than 2^31 - 1 staging work items");
  auto packed_rows = [&](const std::vector<int64_t>& pre) {
    std::vector<int> cnt((size_t)nc);
    std::vector<int64_t> off((size_t)nc);
    for (int64_t k = 0; k < nc; ++k) {
      cnt[k] = (int)(pre[c0 + k + 1] - pre[c0 + k]);
      off[k] = pre[c0 + k] - pre[c0];
    }
    return PackedRows{desc.put(cnt), desc.put(off)};
  };
  h.frames = packed_rows(b.F);
  h.wins = packed_rows(b.Wo);
  if (b.change_out) {
    std::vector<int64_t> off((size_t)nc);
    for (int64_t k = 0; k < nc; ++k) off[k] = k * h.cv.pitch;
    if ((rc = filter_route(b.change_out, nc, off.data(), b.T.data() + c0, off.data(), h.fv))) return rc;
  }
  const SosArgs* filt = b.amp_filt ? &b.amp_sos : nullptr;
  if (b.want_amp && b.env_prm->method == MMF_ENV_HILBERT)
    hilbert_env_route(c0, c1, b.offsets, b.offsets[c0], b.A.data(), filt, h.env);
  else if (b.want_amp && envelope_route(c0, c1, b.offsets, b.offsets[c0], b.geom, b.env_prm->center, b.A.data(), filt,
                                        h.env) < 0)
    return fail(MMF_ERR_UNSUPPORTED, "a chunk of more than 2^31 - 1 envelope work items");
  return MMF_OK;
}

static HostSlot layout_slot(const PackedBatch& b, const HostChunk& h, int nm) {
  const size_t nc = (size_t)(h.c1 - h.c0), pitch = (size_t)h.cv.pitch, W = (size_t)h.mv.W;
  const size_t frames = (size_t)(b.F[h.c1] - b.F[h.c0]), wins = (size_t)(b.Wo[h.c1] - b.Wo[h.c0]);
  const bool mod_c = h.mv.W > 0;
  HostSlot s;
  size_t& o = s.end;
  s.h2d = ws_take(o, (size_t)(b.offsets[h.c1] - b.offsets[h.c0]) * b.isz);
  s.pcm = ws_take(o, nc * h.stride * 4);
  s.tot = ws_take(o, nc * pitch * 8);
  s.mfcc = b.need_mfcc_dev ? ws_take(o, nc * nm * pitch * 4) : 0;
  s.delta = b.delta ? ws_take(o, nc * nm * pitch * 4) : 0;
  s.mag = mod_c && b.mag ? ws_take(o, nc * nm * W * b.nb * 4) : 0;
  s.band = mod_c && b.nbe > 0 ? ws_take(o, nc * W * b.nbe * 4) : 0;
  s.ptot = ws_take(o, frames * 8);
  s.pmfcc = b.mfcc ? ws_take(o, nm * frames * 4) : 0;
  s.pdelta = b.delta ? ws_take(o, nm * frames * 4) : 0;
  s.pmag = mod_c && b.mag ? ws_take(o, nm * wins * b.nb * 4) : 0;
  s.pband = mod_c && b.nbe > 0 ? ws_take(o, wins * b.nbe * 4) : 0;
  s.scratch = ws_take(o, std::max(h.cv.bytes, mod_c ? h.mv.bytes : 0));
  s.amp = b.want_amp ? ws_take(o, (size_t)(b.A[h.c1] - b.A[h.c0]) * 4) : 0;
  s.amp_filt = b.amp_filt ? ws_take(o, (size_t)(b.A[h.c1] - b.A[h.c0]) * 8) : 0;
  s.ctot = b.change_out ? ws_take(o, nc * pitch * 8) : 0;
  s.cwork = b.change_out ? ws_take(o, (size_t)h.fv.work * 8) : 0;
  return s;
}

// Stage 2 (host only): the chunks, each routed, its descriptors appended to `desc` and its slot laid out; `slot`:
// the largest.  Chunk policy: maximal runs of consecutive clips whose samples as they cross PCIe stay within the
// chunk budget (bytes of float32 samples) and whose staged rows at the plan's rate stay within twice that, so that one
// long clip among short ones cannot inflate the padded intermediates.  A clip over either budget is a chunk alone.
static int plan_chunks(const mmf_plan* plan, const PackedBatch& b, std::vector<HostChunk>& chunks, DescBlob& desc,
                       size_t& slot) {
  const int64_t budget = (int64_t)(b.pcm16 ? kHostChunkI16 : kHostChunkF32);
  for (int64_t c0 = 0; c0 < b.n_clips;) {
    int64_t c1 = c0 + 1, n_max = b.len[c0];
    // (at most 65535 clips: the compaction's one CTA per row stays far inside the grid limit)
    while (c1 < b.n_clips && c1 - c0 < 65535) {
      const int64_t m = std::max(n_max, b.len[c1]);
      if ((b.offsets[c1 + 1] - b.offsets[c0]) * 4 > budget || (c1 + 1 - c0) * ((m + 3) & ~3LL) * 4 > 2 * budget)
        break;
      n_max = m;
      ++c1;
    }
    chunks.push_back({c0, c1, (n_max + 3) & ~3LL});
    HostChunk& h = chunks.back();
    if (const int rc = route_chunk(plan, b, h, desc)) return rc;
    h.slot = layout_slot(b, h, plan->cfg.n_mfcc);
    slot = std::max(slot, h.slot.end);
    c0 = c1;
  }
  // then every chunk's stage descriptors (mostly chunk tables), copied once into one allocation
  size_t bytes = desc.size();
  for (const HostChunk& h : chunks)
    bytes += 4 * kDescAlign + h.cv.desc.size() + h.mv.desc.size() + h.env.desc.size() + h.fv.desc.size();
  desc.bytes.reserve(bytes);
  for (HostChunk& h : chunks) {
    h.o_cv = desc.put(h.cv.desc.bytes);
    h.o_mv = desc.put(h.mv.desc.bytes);
    h.o_env = desc.put(h.env.desc.bytes);
    h.o_fv = desc.put(h.fv.desc.bytes);
  }
  slot = align_up(slot, 256);
  return MMF_OK;
}

// Stage 3: one chunk's device sequence on `st`.  One H2D copy of its packed samples; the envelope, read from the
// native samples as they arrived; the staging launch into rows at the plan's rate; the change and modulation stages;
// then per output one compaction (padded rows -> packed blocks) and one D2H copy.  dd: the call's descriptors on the
// device, taps: the tap table there; base: the chunk's slot.
static int run_chunk(mmf_plan* plan, const PackedBatch& b, const HostChunk& h, const unsigned char* dd,
                     const float* taps, unsigned char* base, cudaStream_t st) {
  const int64_t nc = h.c1 - h.c0;
  const int nm = plan->cfg.n_mfcc;
  const HostSlot& s = h.slot;
  auto dev = [&](size_t o) { return (void*)(base + o); };
  MMF_CUDA(cudaMemcpyAsync(dev(s.h2d), (const unsigned char*)b.pcm + (size_t)b.offsets[h.c0] * b.isz,
                           (size_t)(b.offsets[h.c1] - b.offsets[h.c0]) * b.isz, cudaMemcpyHostToDevice, st));
  float* d_amp = b.want_amp ? (float*)dev(s.amp) : nullptr;
  double* d_ampf = b.amp_filt ? (double*)dev(s.amp_filt) : nullptr;
  int rc;
  if (b.want_amp &&
      (rc = envelope_run(h.env, dd + h.o_env, dev(s.h2d), b.pcm16, d_amp, d_ampf, plan->sm_count, st)))
    return rc;
  float* d_pcm = (float*)dev(s.pcm);
  cudaError_t e = resample_rows_launch(dev(s.h2d), b.pcm16, (const RsClip*)(dd + h.stage.clips),
                                       (const unsigned*)(dd + h.stage.first), (long)nc, (long)h.stage.items, taps,
                                       d_pcm, (long)h.stride, st);
  if (e != cudaSuccess) return cuda_fail(e, "resample_rows_kernel launch");
  double* d_tot = (double*)dev(s.tot);
  float* d_mfcc = b.need_mfcc_dev ? (float*)dev(s.mfcc) : nullptr;
  float* d_delta = b.delta ? (float*)dev(s.delta) : nullptr;
  if ((rc = change_varlen_run(plan, h.cv, base + s.scratch, dd + h.o_cv, d_pcm, h.stride, b.prm, d_tot, nullptr,
                              d_mfcc, d_delta, st)))
    return rc;
  if (b.change_out) {  // the raw curves -> their own rows, which the compaction then reads
    double* d_ctot = (double*)dev(s.ctot);
    if ((rc = filter_run(b.change_out, h.fv, dd + h.o_fv, d_tot, 0, d_ctot, (double*)dev(s.cwork), st))) return rc;
    d_tot = d_ctot;
  }
  const bool mod_c = h.mv.W > 0;
  float* d_mag = mod_c && b.mag ? (float*)dev(s.mag) : nullptr;
  float* d_band = mod_c && b.nbe > 0 ? (float*)dev(s.band) : nullptr;
  if (mod_c && (rc = modspec_varlen_run(plan, h.mv, base + s.scratch, dd + h.o_mv, d_mfcc, nm, h.cv.pitch,
                                        b.mod->win, b.mod->hop, b.mod->nfft, d_mag, d_band, st)))
    return rc;
  // one requested output (host != null): padded rows -> packed blocks in the slot -> one copy back
  const long pitch = h.cv.pitch, W = (long)h.mv.W;
  auto out = [&](const void* src, size_t o_dst, int eb, int rows, int unit, long pitch_el, bool per_win,
                 void* host) -> int {
    const int64_t* pre = per_win ? b.Wo.data() : b.F.data();
    const size_t blk = (size_t)eb * rows * unit, n = (size_t)(pre[h.c1] - pre[h.c0]);
    if (!host || !n) return MMF_OK;
    const PackedRows& pr = per_win ? h.wins : h.frames;
    cudaError_t ce = compact_rows_launch(src, dev(o_dst), eb, (long)nc, rows, unit, pitch_el,
                                         (const int*)(dd + pr.cnt), (const long*)(dd + pr.off), st);
    if (ce != cudaSuccess) return cuda_fail(ce, "compact_rows_kernel launch");
    MMF_CUDA(cudaMemcpyAsync((char*)host + blk * pre[h.c0], dev(o_dst), blk * n, cudaMemcpyDeviceToHost, st));
    return MMF_OK;
  };
  if ((rc = out(d_tot, s.ptot, 8, 1, 1, pitch, false, b.tot)) ||
      (rc = out(d_mfcc, s.pmfcc, 4, nm, 1, pitch, false, b.mfcc)) ||
      (rc = out(d_delta, s.pdelta, 4, nm, 1, pitch, false, b.delta)) ||
      (rc = out(d_mag, s.pmag, 4, nm, b.nb, W * b.nb, true, d_mag ? b.mag : nullptr)) ||
      (rc = out(d_band, s.pband, 4, 1, b.nbe, W * b.nbe, true, d_band ? b.band : nullptr)))
    return rc;
  const size_t n_amp = b.want_amp ? (size_t)(b.A[h.c1] - b.A[h.c0]) : 0;
  if (b.amp) MMF_CUDA(cudaMemcpyAsync(b.amp + b.A[h.c0], d_amp, n_amp * 4, cudaMemcpyDeviceToHost, st));
  if (d_ampf) MMF_CUDA(cudaMemcpyAsync(b.amp_filt + b.A[h.c0], d_ampf, n_amp * 8, cudaMemcpyDeviceToHost, st));
  return MMF_OK;
}

// The packed host-buffer bundle: the host-only checks, the chunk plan, then each chunk's device sequence
static int features_host_varlen_impl(mmf_plan* plan, PackedBatch b) {
  int rc = packed_check(plan, b);
  if (rc) return rc;
  // every chunk is routed before anything is queued; the call's descriptors: the taps, then each chunk's
  DescBlob desc;
  const size_t o_taps = desc.put(b.h_taps, (size_t)b.n_taps);
  std::vector<HostChunk> chunks;
  size_t slot = 0;
  if ((rc = plan_chunks(plan, b, chunks, desc, slot))) return rc;
  // the change curves' output filter: checked after every clip passed the change stage's own length checks
  for (int64_t i = 0; b.change_out && i < b.n_clips; ++i)
    if ((rc = filter_row_check(b.change_out, b.T[i], i))) return rc;
  MMF_CUDA(cudaSetDevice(plan->cfg.device));
  const size_t o_slots = align_up(desc.size(), 256);
  if ((rc = ensure_host_ws(plan, o_slots + 2 * slot))) return rc;
  // the modulation tables are (re)built with a device-wide synchronisation: do it before any copy is queued
  if (b.want_mod && b.Wo[b.n_clips] > 0 &&
      (rc = ensure_mod_tables(plan, b.mod->win, b.mod->nfft, b.mod->band_lo, b.mod->band_hi, b.nbe)))
    return rc;
  return run_and_drain(plan, [&]() -> int {
    // every chunk's descriptors go up in one copy, complete before either stream reads them: a copy from pageable
    // memory waits for its stream, so inside the loop it would hold back the next chunk's queueing
    unsigned char* d_desc = (unsigned char*)plan->host_ws;
    MMF_CUDA(cudaMemcpyAsync(d_desc, desc.bytes.data(), desc.size(), cudaMemcpyHostToDevice, plan->streams[0]));
    MMF_CUDA(cudaStreamSynchronize(plan->streams[0]));
    // stream order serialises reuse of slot k & 1 (chunk k - 2 ran on the same stream)
    for (size_t k = 0; k < chunks.size(); ++k)
      if (const int rc2 = run_chunk(plan, b, chunks[k], d_desc, (const float*)(d_desc + o_taps),
                                    d_desc + o_slots + (k & 1) * slot, plan->streams[k & 1]))
        return rc2;
    return MMF_OK;
  });
}

}  // namespace mmf

extern "C" {

int mmf_features_varlen_sizes(const mmf_config* cfg, const mmf_modspec_params* mod, int64_t n_clips,
                              const int64_t* offsets_host, int64_t* frame_off_host, int64_t* win_off_host) {
  using namespace mmf;
  int rc = validate_offsets(n_clips, offsets_host);
  if (rc) return rc;
  if (!cfg || !frame_off_host || !win_off_host) return fail(MMF_ERR_INVALID, "NULL argument");
  if (cfg->n_fft < 1 || cfg->hop_length < 1) return fail(MMF_ERR_INVALID, "need n_fft >= 1 and hop_length >= 1");
  const bool windows = mod && mod->win > 0;
  if (windows && mod->hop < 1) return fail(MMF_ERR_INVALID, "modulation hop must be >= 1");
  packed_sizes(cfg->n_fft, cfg->hop_length, windows ? mod->win : 0, windows ? mod->hop : 1, n_clips, offsets_host,
               frame_off_host, win_off_host);
  return MMF_OK;
}

int mmf_features_host_varlen(mmf_plan* plan, const float* pcm_host, int64_t n_clips, const int64_t* offsets_host,
                             const mmf_change_params* prm, const mmf_modspec_params* mod, double* tot_host,
                             float* mfcc_host, float* delta_host, float* mag_host, float* band_host) {
  return mmf::features_host_varlen_impl(plan, {pcm_host, 0, n_clips, offsets_host, nullptr, nullptr, 0, prm, mod,
                                               nullptr, nullptr, tot_host, mfcc_host, delta_host, mag_host, band_host});
}

int mmf_features_host_varlen_resampled(mmf_plan* plan, const void* pcm_host, int32_t pcm16, int64_t n_clips,
                                       const int64_t* offsets_host, const mmf_resample_clip* rs_host,
                                       const float* h_host, int64_t n_h, const mmf_change_params* prm,
                                       const mmf_modspec_params* mod, double* tot_host, float* mfcc_host,
                                       float* delta_host, float* mag_host, float* band_host) {
  return mmf::features_host_varlen_impl(plan, {pcm_host, pcm16 ? 1 : 0, n_clips, offsets_host, rs_host, h_host, n_h,
                                               prm, mod, nullptr, nullptr, tot_host, mfcc_host, delta_host, mag_host,
                                               band_host, nullptr, nullptr, true});
}

int mmf_features_host_varlen_pcm16(mmf_plan* plan, const int16_t* pcm16_host, int64_t n_clips,
                                   const int64_t* offsets_host, const mmf_change_params* prm,
                                   const mmf_modspec_params* mod, double* tot_host, float* mfcc_host,
                                   float* delta_host, float* mag_host, float* band_host) {
  return mmf::features_host_varlen_impl(plan, {pcm16_host, 1, n_clips, offsets_host, nullptr, nullptr, 0, prm, mod,
                                               nullptr, nullptr, tot_host, mfcc_host, delta_host, mag_host, band_host});
}

int mmf_features_host_varlen_out(mmf_plan* plan, const void* pcm_host, int32_t pcm16, int64_t n_clips,
                                 const int64_t* offsets_host, const mmf_resample_clip* rs_host, const float* h_host,
                                 int64_t n_h, const mmf_change_params* prm, const mmf_modspec_params* mod,
                                 const mmf_env_params* env, const int32_t* geom_host,
                                 const mmf_out_filter* change_out, double* tot_host, float* mfcc_host,
                                 float* delta_host, float* mag_host, float* band_host, float* amp_host,
                                 double* amp_filt_host) {
  return mmf::features_host_varlen_impl(plan, {pcm_host, pcm16 ? 1 : 0, n_clips, offsets_host, rs_host, h_host, n_h,
                                               prm, mod, env, geom_host, tot_host, mfcc_host, delta_host, mag_host,
                                               band_host, amp_host, amp_filt_host, rs_host != nullptr, change_out});
}

int mmf_features_host_varlen_env(mmf_plan* plan, const void* pcm_host, int32_t pcm16, int64_t n_clips,
                                 const int64_t* offsets_host, const mmf_resample_clip* rs_host, const float* h_host,
                                 int64_t n_h, const mmf_change_params* prm, const mmf_modspec_params* mod,
                                 const mmf_env_params* env, const int32_t* geom_host, double* tot_host,
                                 float* mfcc_host, float* delta_host, float* mag_host, float* band_host,
                                 float* amp_host, double* amp_filt_host) {
  return mmf_features_host_varlen_out(plan, pcm_host, pcm16, n_clips, offsets_host, rs_host, h_host, n_h, prm, mod,
                                      env, geom_host, nullptr, tot_host, mfcc_host, delta_host, mag_host, band_host,
                                      amp_host, amp_filt_host);
}

int mmf_features_host_varlen_amp(mmf_plan* plan, const void* pcm_host, int32_t pcm16, int64_t n_clips,
                                 const int64_t* offsets_host, const mmf_resample_clip* rs_host, const float* h_host,
                                 int64_t n_h, const mmf_change_params* prm, const mmf_modspec_params* mod,
                                 const mmf_amp_params* amp, const int32_t* geom_host, double* tot_host,
                                 float* mfcc_host, float* delta_host, float* mag_host, float* band_host,
                                 float* amp_host, double* amp_filt_host) {
  mmf_env_params env{};
  if (amp) {
    env.method = MMF_ENV_RMS;
    env.center = amp->center;
    env.out_n_sections = amp->out_n_sections;
    std::memcpy(env.out_sos, amp->out_sos, sizeof(env.out_sos));
  }
  return mmf_features_host_varlen_env(plan, pcm_host, pcm16, n_clips, offsets_host, rs_host, h_host, n_h, prm, mod,
                                      amp ? &env : nullptr, geom_host, tot_host, mfcc_host, delta_host, mag_host,
                                      band_host, amp_host, amp_filt_host);
}

int mmf_env_varlen_sizes(int64_t n_clips, const int64_t* offsets_host, const mmf_env_params* env,
                         const int32_t* geom_host, int64_t* amp_off_host) {
  using namespace mmf;
  int rc = validate_offsets(n_clips, offsets_host);
  if (rc) return rc;
  if (!env || !amp_off_host) return fail(MMF_ERR_INVALID, "env and amp_off_host must not be NULL");
  return env_sizes(n_clips, offsets_host, env, geom_host, amp_off_host);
}

int mmf_hilbert_varlen(mmf_plan* plan, const float* x_dev, int64_t n_clips, const int64_t* offsets_host,
                       float* amp_dev, void* stream) {
  using namespace mmf;
  int rc = validate_offsets(n_clips, offsets_host);
  if (rc) return rc;
  mmf_env_params env{};
  env.method = MMF_ENV_HILBERT;
  std::vector<int64_t> A((size_t)n_clips + 1);
  if ((rc = env_sizes(n_clips, offsets_host, &env, nullptr, A.data()))) return rc;
  if (!plan || !x_dev || !amp_dev) return fail(MMF_ERR_INVALID, "NULL argument");
  EnvelopeVarlen v;
  hilbert_env_route(0, n_clips, offsets_host, 0, A.data(), nullptr, v);
  return rms_run(plan, x_dev, v, amp_dev, (cudaStream_t)stream);
}

int mmf_amp_varlen_sizes(int64_t n_clips, const int64_t* offsets_host, const int32_t* geom_host, int32_t center,
                         int64_t* amp_off_host) {
  using namespace mmf;
  int rc = validate_offsets(n_clips, offsets_host);
  if (rc) return rc;
  if (!amp_off_host) return fail(MMF_ERR_INVALID, "amp_off_host is NULL");
  return amp_sizes(n_clips, offsets_host, geom_host, center, amp_off_host);
}

int mmf_rms_varlen(mmf_plan* plan, const float* x_dev, int64_t n_clips, const int64_t* offsets_host,
                   const int32_t* geom_host, int32_t center, float* amp_dev, void* stream) {
  using namespace mmf;
  int rc = validate_offsets(n_clips, offsets_host);
  if (rc) return rc;
  std::vector<int64_t> A((size_t)n_clips + 1);
  if ((rc = amp_sizes(n_clips, offsets_host, geom_host, center, A.data()))) return rc;
  if (!plan || !x_dev || !amp_dev) return fail(MMF_ERR_INVALID, "NULL argument");
  EnvelopeVarlen v;
  if (envelope_route(0, n_clips, offsets_host, 0, geom_host, center, A.data(), nullptr, v) < 0)
    return fail(MMF_ERR_UNSUPPORTED, "more than 2^31 - 1 work items");
  return rms_run(plan, x_dev, v, amp_dev, (cudaStream_t)stream);
}

}  // extern "C"

extern "C" {

int mmf_features_host(mmf_plan* plan, const float* pcm_host, int64_t n_clips, int64_t n_samples, int64_t clip_stride,
                      const mmf_change_params* prm, const mmf_modspec_params* mod, double* tot_host, float* mfcc_host,
                      float* delta_host, float* mag_host, float* band_host) {
  return features_host_impl(plan, pcm_host, 0, n_clips, n_samples, clip_stride, prm, mod, tot_host, mfcc_host,
                            delta_host, mag_host, band_host);
}

int mmf_features_host_pcm16(mmf_plan* plan, const int16_t* pcm16_host, int64_t n_clips, int64_t n_samples,
                            int64_t clip_stride, const mmf_change_params* prm, const mmf_modspec_params* mod,
                            double* tot_host, float* mfcc_host, float* delta_host, float* mag_host,
                            float* band_host) {
  return features_host_impl(plan, pcm16_host, 1, n_clips, n_samples, clip_stride, prm, mod, tot_host, mfcc_host,
                            delta_host, mag_host, band_host);
}

int mmf_hilbert_envelope(mmf_plan* plan, const float* x_dev, int64_t n_clips, int64_t n, int64_t x_stride,
                         float* amp_dev, int64_t amp_stride, void* stream) {
  if (!plan || !x_dev || !amp_dev) return fail(MMF_ERR_INVALID, "NULL argument");
  if (n_clips < 1 || n < 1 || n > (1L << 26)) return fail(MMF_ERR_UNSUPPORTED, "need 1 <= n <= 2^26 samples");
  MMF_CUDA(cudaSetDevice(plan->cfg.device));
  if (n > kHilDirectMax) {
    // O(n log n): the rows as one ragged batch of Bluestein transforms (hilbert_fft.cu)
    EnvelopeVarlen v;
    v.method = MMF_ENV_HILBERT;
    v.n_clips = n_clips;
    std::vector<long> src((size_t)n_clips), len((size_t)n_clips, (long)n), out((size_t)n_clips);
    for (int64_t i = 0; i < n_clips; ++i) {
      src[i] = (long)(i * x_stride);
      out[i] = (long)(i * amp_stride);
    }
    hilbert_route(src, len, out, v.hil, v.desc);
    return rms_run(plan, x_dev, v, amp_dev, (cudaStream_t)stream);
  }
  // short signals: the equivalent circular convolution with the discrete Hilbert kernel, evaluated directly
  const cudaError_t e = hilbert_envelope_launch(x_dev, 0, n_clips, n, x_stride, amp_dev, amp_stride, plan->sm_count,
                                                (cudaStream_t)stream);
  if (e != cudaSuccess) return cuda_fail(e, "hilbert kernels launch");
  return MMF_OK;
}

int mmf_find_peaks(mmf_plan* plan, const double* x_dev, int64_t rows, int64_t T, int64_t row_stride, int32_t minima,
                   int32_t max_peaks, int32_t* idx_dev, int32_t* count_dev, void* stream) {
  if (!plan || !x_dev || !idx_dev || !count_dev) return fail(MMF_ERR_INVALID, "NULL argument");
  if (rows < 1 || T < 1 || max_peaks < 1 || rows > (1L << 26)) return fail(MMF_ERR_INVALID, "bad sizes");
  MMF_CUDA(cudaSetDevice(plan->cfg.device));
  cudaError_t e = find_peaks_launch(x_dev, rows, T, row_stride, minima, max_peaks, idx_dev, count_dev,
                                    (cudaStream_t)stream);
  if (e != cudaSuccess) return cuda_fail(e, "find_peaks_kernel launch");
  return MMF_OK;
}

int mmf_pcm16_to_f32(mmf_plan* plan, const int16_t* pcm16_dev, int64_t n, float* pcm_dev, void* stream) {
  if (!plan || !pcm16_dev || !pcm_dev) return fail(MMF_ERR_INVALID, "NULL argument");
  if (n < 1) return fail(MMF_ERR_INVALID, "n must be positive");
  MMF_CUDA(cudaSetDevice(plan->cfg.device));
  cudaError_t e = pcm16_to_f32_launch(pcm16_dev, n, pcm_dev, (cudaStream_t)stream);
  if (e != cudaSuccess) return cuda_fail(e, "pcm16_to_f32_kernel launch");
  return MMF_OK;
}

int mmf_resample_poly(mmf_plan* plan, const float* x_dev, int64_t n_clips, int64_t n_in, int64_t x_stride,
                      const float* h_host, int32_t len_h, int32_t up, int32_t down, int64_t n_pre_remove, int64_t n_out,
                      float* y_dev, int64_t y_stride, void* stream) {
  if (!plan || !x_dev || !h_host || !y_dev) return fail(MMF_ERR_INVALID, "NULL argument");
  if (n_clips < 1 || n_clips > 65535 || n_in < 1 || n_out < 1) return fail(MMF_ERR_INVALID, "bad sizes");
  if (up < 1 || down < 1 || len_h < 1 || len_h > (1 << 22))
    return fail(MMF_ERR_UNSUPPORTED, "need up, down >= 1 and a filter of at most 2^22 taps");
  if ((n_out + kRsOut - 1) / kRsOut * n_clips > 0x7fffffffLL) return fail(MMF_ERR_UNSUPPORTED, "too many outputs");
  // one descriptor per row, all reading the one filter (up = down = 1 filters too: nothing here is a copy)
  std::vector<RsClip> cl((size_t)n_clips);
  std::vector<unsigned> first((size_t)n_clips + 1);
  const int64_t per = (n_out + kRsOut - 1) / kRsOut;
  for (int64_t r = 0; r < n_clips; ++r) {
    cl[r] = RsClip{(long)(r * x_stride), (long)n_in, (long)n_pre_remove, (long)n_out, 0, up, down, len_h, 0};
    first[r] = (unsigned)(r * per);
  }
  first[n_clips] = (unsigned)(n_clips * per);
  DescBlob desc;
  const RaggedParts p{desc.put(cl), desc.put(first), n_clips * per};
  return resample_dev(plan, x_dev, desc, p, h_host, len_h, n_clips, y_dev, y_stride, (cudaStream_t)stream);
}

int mmf_resample_varlen(mmf_plan* plan, const float* x_dev, int64_t n_clips, const int64_t* offsets_host,
                        const mmf_resample_clip* rs_host, const float* h_host, int64_t n_h, float* y_dev,
                        int64_t y_stride, void* stream) {
  int rc = validate_offsets(n_clips, offsets_host);
  int64_t n_taps = 0;
  if (rc || (rc = validate_resample(n_clips, offsets_host, rs_host, h_host, n_h, &n_taps))) return rc;
  if (!plan || !x_dev || !y_dev) return fail(MMF_ERR_INVALID, "NULL argument");
  for (int64_t i = 0; i < n_clips; ++i)
    if (rs_host[i].n_out > y_stride) {
      char buf[128];
      std::snprintf(buf, sizeof(buf), "clip %lld: n_out %lld exceeds y_stride %lld", (long long)i,
                    (long long)rs_host[i].n_out, (long long)y_stride);
      return fail(MMF_ERR_INVALID, buf);
    }
  DescBlob desc;
  const RaggedParts p = resample_desc(0, n_clips, offsets_host, 0, rs_host, desc);
  if (p.items < 0) return fail(MMF_ERR_UNSUPPORTED, "more than 2^31 - 1 work items");
  return resample_dev(plan, x_dev, desc, p, h_host, n_taps, n_clips, y_dev, y_stride, (cudaStream_t)stream);
}

// the single-row-type calls: one descriptor per row of the ragged kernels (the 65 535-row limit is theirs)
int mmf_fir_filtfilt(mmf_plan* plan, const double* x_dev, int64_t rows, int64_t T, const double* b_host,
                     int32_t n_taps, double* y_dev, double* work_dev, void* stream) {
  if (!plan || !x_dev || !b_host || !y_dev || !work_dev) return fail(MMF_ERR_INVALID, "NULL argument");
  if (n_taps < 1 || n_taps > 4096) return fail(MMF_ERR_UNSUPPORTED, "n_taps must be in [1, 4096]");
  if (rows < 1 || rows > 65535) return fail(MMF_ERR_UNSUPPORTED, "rows must be in [1, 65535]");
  if (T <= 3 * n_taps) return too_short(3 * n_taps);
  mmf_out_filter f{};
  f.kind = MMF_FILT_FIR;
  f.n_taps = n_taps;
  f.taps = b_host;
  std::vector<int64_t> off((size_t)rows), len((size_t)rows, T);
  for (int64_t r = 0; r < rows; ++r) off[r] = r * T;
  FilterVarlen v;
  int rc = filter_route(&f, rows, off.data(), len.data(), off.data(), v);
  if (rc) return rc;
  // work_dev [rows, T + 6 * n_taps] is the forward pass's scratch, packed as filter_route packs it
  return filter_uploaded(plan, &f, v, x_dev, 0, y_dev, work_dev, (cudaStream_t)stream);
}

int mmf_stencil(mmf_plan* plan, const double* x_dev, int64_t rows, int64_t T, const double* coef_host, int32_t half,
                const double* edge_l_host, const double* edge_r_host, int32_t n_edge, int32_t n_edge_in,
                double* y_dev, void* stream) {
  if (!plan || !x_dev || !coef_host || !y_dev) return fail(MMF_ERR_INVALID, "NULL argument");
  if (half < 0 || n_edge < half || n_edge_in < 0) return fail(MMF_ERR_INVALID, "need n_edge >= half >= 0");
  if (n_edge > 0 && (!edge_l_host || !edge_r_host)) return fail(MMF_ERR_INVALID, "edge matrices are NULL");
  if (T < n_edge_in || T < 2 * n_edge) return fail(MMF_ERR_TOO_SHORT, "input shorter than the stencil's edge window");
  if (rows < 1 || rows > 65535) return fail(MMF_ERR_UNSUPPORTED, "rows must be in [1, 65535]");
  if (T < 1) return fail(MMF_ERR_INVALID, "T must be positive");
  mmf_out_filter f{};
  f.kind = MMF_FILT_SG;
  f.half = half;
  f.coef = coef_host;
  f.n_edge = n_edge;
  f.n_edge_in = n_edge_in;
  f.edge_l = edge_l_host;
  f.edge_r = edge_r_host;
  std::vector<int64_t> off((size_t)rows), len((size_t)rows, T);
  for (int64_t r = 0; r < rows; ++r) off[r] = r * T;
  FilterVarlen v;
  int rc = filter_route(&f, rows, off.data(), len.data(), off.data(), v);
  if (rc) return rc;
  return filter_uploaded(plan, &f, v, x_dev, 0, y_dev, nullptr, (cudaStream_t)stream);
}

int mmf_filter_varlen_check(const mmf_out_filter* filt, int64_t n_rows, const int64_t* T_host) {
  int rc = filter_shape_check(filt);
  if (rc) return rc;
  if (n_rows < 1) return fail(MMF_ERR_INVALID, "n_rows must be positive");
  if (!T_host) return fail(MMF_ERR_INVALID, "T_host is NULL");
  for (int64_t i = 0; i < n_rows; ++i) {
    if (T_host[i] < 1) return fail(MMF_ERR_INVALID, "clip " + std::to_string(i) + ": T must be positive");
    if ((rc = filter_row_check(filt, T_host[i], i))) return rc;
  }
  return MMF_OK;
}

int mmf_filter_varlen(mmf_plan* plan, const mmf_out_filter* filt, const void* x_dev, int32_t x_is_f32, int64_t n_rows,
                      const int64_t* x_off_host, const int64_t* T_host, double* y_dev, const int64_t* y_off_host,
                      void* stream) {
  int rc = mmf_filter_varlen_check(filt, n_rows, T_host);
  if (rc) return rc;
  if (!plan || !x_dev || !y_dev || !x_off_host || !y_off_host) return fail(MMF_ERR_INVALID, "NULL argument");
  FilterVarlen v;
  if ((rc = filter_route(filt, n_rows, x_off_host, T_host, y_off_host, v))) return rc;
  return filter_uploaded(plan, filt, v, x_dev, x_is_f32 ? 1 : 0, y_dev, nullptr, (cudaStream_t)stream);
}

// one descriptor per row of the ragged kernel (rows of equal length: the grid has no row limit)
int mmf_rms(mmf_plan* plan, const float* pcm_dev, int64_t n_clips, int64_t n_samples, int64_t clip_stride,
            int32_t frame_length, int32_t hop_length, int32_t center, float* rms_dev, void* stream) {
  if (!plan || !pcm_dev || !rms_dev) return fail(MMF_ERR_INVALID, "NULL argument");
  if (n_clips < 1) return fail(MMF_ERR_INVALID, "n_clips must be positive");
  if (frame_length < 1 || hop_length < 1) return fail(MMF_ERR_INVALID, "frame_length and hop_length must be positive");
  const int pad = center ? frame_length / 2 : 0;
  const int64_t padded = n_samples + 2 * (int64_t)pad;
  if (padded < frame_length) return fail(MMF_ERR_TOO_SHORT, "Input is too short for frame_length");
  const int64_t T = 1 + (padded - frame_length) / hop_length;
  const int F = rms_frames_per_item(frame_length, hop_length);
  const int64_t per = (T + F - 1) / F;
  if (per * n_clips > 0x7fffffffLL) return fail(MMF_ERR_UNSUPPORTED, "more than 2^31 - 1 work items");
  std::vector<RmsClip> cl((size_t)n_clips);
  std::vector<unsigned> first((size_t)n_clips + 1);
  for (int64_t r = 0; r < n_clips; ++r) {
    cl[r] = RmsClip{(long)(r * clip_stride), (long)n_samples, (long)(r * T), (long)T, frame_length, hop_length, pad, F};
    first[r] = (unsigned)(r * per);
  }
  first[n_clips] = (unsigned)(n_clips * per);
  EnvelopeVarlen v;
  v.n_clips = n_clips;
  v.rms = RaggedParts{v.desc.put(cl), v.desc.put(first), n_clips * per};
  return rms_run(plan, pcm_dev, v, rms_dev, (cudaStream_t)stream);
}

int mmf_mfcc_change_host(mmf_plan* plan, const float* pcm_host, int64_t n_clips, int64_t n_samples,
                         int64_t clip_stride, const mmf_change_params* prm, double* tot_host, float* mfcc_host) {
  return mmf_features_host(plan, pcm_host, n_clips, n_samples, clip_stride, prm, nullptr, tot_host, mfcc_host, nullptr,
                           nullptr, nullptr);
}

}  // extern "C"
