// C ABI of libdspfront.so (include/dspfront.h): context, planning, host staging pipeline and
// the launch logic that routes a batch to the int16 fast kernel (frontend_pcm.cu) with the
// float64 replay kernel (frontend_exact.cu) behind it.  No CPU implementation lives here:
// host code only plans, copies and launches.
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <iterator>
#include <memory>
#include <string>
#include <utility>
#include <vector>

#include "kernels.cuh"
#include "knn.cuh"
#include "mfcc_dtw.cuh"
#include "misc.cuh"

using namespace dsp;

namespace {

thread_local std::string g_err;

int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}

#define CU(expr)                                                                         \
  do {                                                                                   \
    cudaError_t e__ = (expr);                                                            \
    if (e__ != cudaSuccess)                                                              \
      return fail(DSP_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), \
                  __FILE__, __LINE__);                                                   \
  } while (0)

// Owners of the library's device memory, pinned memory, streams and events: each one frees what it holds when it is
// destroyed, so a handle or table entry releases everything with it, on an error return too.  Every destruction keeps
// two rules:
//  - the owner's device is current: dsp_destroy, dsp_knn_free and dsp_dtw_free call cudaSetDevice first, and every
//    other destruction happens inside an entry point that has already set the device;
//  - no queued work still uses it: those three synchronise before they free, and the window / MFCC table caches are
//    emptied only after cudaDeviceSynchronize.
// Host vectors that are sources of stream-ordered copies (MfccEntry::win / tw / range, dsp_dtw::h_len) belong to the
// owner of the device buffers they fill, so they live as long as those buffers.
template <bool kPinned>
struct Buf {
  void* p = nullptr;
  size_t cap = 0;
  Buf() = default;
  Buf(const Buf&) = delete;
  Buf& operator=(const Buf&) = delete;
  Buf(Buf&& o) noexcept : p(o.p), cap(o.cap) { o.p = nullptr; o.cap = 0; }
  Buf& operator=(Buf&& o) noexcept { std::swap(p, o.p); std::swap(cap, o.cap); return *this; }
  ~Buf() { reset(); }
  // device buffers grow with 1/8 headroom, pinned staging buffers by 256 bytes
  cudaError_t ensure(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    reset();
    const size_t want = kPinned ? bytes + 256 : bytes + bytes / 8 + 256;
    const cudaError_t e = kPinned ? cudaMallocHost(&p, want) : cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  template <class T> T* as() const { return reinterpret_cast<T*>(p); }

 private:
  void reset() {
    if (p && kPinned) cudaFreeHost(p);
    if (p && !kPinned) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
};
using DevBuf = Buf<false>;
using PinBuf = Buf<true>;

// a stream or event the library created (dsp_context::stream is not one: it may be the caller's)
template <class T, cudaError_t (*Destroy)(T)>
struct Owned {
  T h = nullptr;
  Owned() = default;
  Owned(const Owned&) = delete;
  Owned& operator=(const Owned&) = delete;
  Owned(Owned&& o) noexcept : h(o.h) { o.h = nullptr; }
  Owned& operator=(Owned&& o) noexcept { std::swap(h, o.h); return *this; }
  ~Owned() { if (h) Destroy(h); }
  operator T() const { return h; }
};
using Stream = Owned<cudaStream_t, cudaStreamDestroy>;
using Event = Owned<cudaEvent_t, cudaEventDestroy>;

constexpr size_t kMaxSmemPerCta = 227 * 1024;
constexpr int64_t kFastMaxLen = 1 << 20;          // exact-integer bounds of the fast kernel
constexpr int kKnnDenseMaxDim = 16384;            // feature dimensions served by the tensor-core scan
constexpr int64_t kKnnDenseQueryChunk = 32768;    // queries packed per scan launch
// candidate scan of a KNN handle, numbered as dsp_knn_last_stats reports it
enum KnnScan { kScanF64 = 0, kScanFp32 = 1, kScanDense = 2, kScanTc16 = 3 };
constexpr size_t kHostChunkBytesDefault = 512u << 20;    // samples per staged chunk of the host pipeline (DSP_HOST_CHUNK_MB overrides): 96 MB 550 k audio-s/s end to end, 512 MB 586 k, 2 GB 592 k (pinned H2D alone: 55.6 GB/s = 630 k)
static size_t host_chunk_bytes() {
  static const size_t v = [] { const char* e = std::getenv("DSP_HOST_CHUNK_MB"); const long mb = e ? std::atol(e) : 0; return mb >= 1 && mb <= 4096 ? (size_t)mb << 20 : kHostChunkBytesDefault; }();
  return v;
}

size_t dtype_size(int dtype) {
  switch (dtype) {
    case DSP_S16: return 2;
    case DSP_U8: return 1;
    case DSP_F32: return 4;
    case DSP_F64: return 8;
    default: return 0;
  }
}

struct Slot {
  DevBuf samples, off, ints, stats, feat, epd_e, epd_z, f64;
  PinBuf h_off;
  Event ev_in, ev_k, ev_out;
};

}  // namespace

struct dsp_context {
  int device = 0;
  int sm_count = 0;
  size_t smem_optin = 0;        // opt-in shared memory per block (227 KB on sm_100), static + dynamic
  Stream own, s_in, s_out;
  cudaStream_t stream = nullptr;
  int64_t launches = 0;
  // window tables stay resident per (type, length): a context that alternates windows (three front ends sharing one
  // context, a sweep over frame lengths) never re-uploads or synchronises, and kernels still running on a previously
  // installed stream keep reading the table they were launched with
  struct WinEntry { int type, len; DevBuf w64, w32; };
  std::vector<std::unique_ptr<WinEntry>> windows;
  const double* win64 = nullptr;
  const float* win32 = nullptr;
  DevBuf counters;   // [0] work counter (u32)  [1] flag count (i32)
  DevBuf flag_list, zbuf, seqbuf;
  DevBuf prof;       // DSP_PROF phase counters of the fast kernels
  size_t occ_smem = 0;
  int occ_variant = -1;
  int pcm_variant = -1;         // -1 automatic; else a build of frontend_pcm.cu's kVariants (dsp_set_tuning / DSP_PCM_VARIANT)
  int stagger_ns = 0;           // DSP_STAGGER_NS (tuning knob)
  int tma_chunk = 4096;         // bytes per bulk copy; DSP_TMA_CHUNK overrides (tuning knob)
  int knn_prune = 1;            // tile pruning of the D <= 15 filter: 0 off, 1 unless the lists keep > 85 % of the tiles, 2 always
  int occ = 0;
  Slot slot[2];
  DevBuf tmp[16];
  // device tables of dsp_mfcc_batch_device, kept per (parameters, filterbank, DCT): a repeated call copies nothing
  struct MfccEntry {
    int frame_length, window, n_fft, n_mels, n_ceps;
    std::vector<float> fb, dct;                 // the caller's tables (the key) ...
    std::vector<float> win, tw;                 // ... and the derived host tables, alive until their copies are done
    std::vector<int> range;
    DevBuf d_win, d_tw, d_fb, d_range, d_dct;
  };
  std::vector<std::unique_ptr<MfccEntry>> mfcc_tables;
  DevBuf mfcc_work;  // work counter of the device MFCC call
};

struct dsp_dtw {
  dsp_context* ctx = nullptr;
  int64_t nt = 0, index_base = 0;
  int dim = 0, k = 0, max_t = 0, warps = 1;
  std::vector<int32_t> h_len;                   // source of the t_len upload
  DevBuf feats, offsets, t_len, labels, cand_d, cand_i, stats;
};

struct dsp_knn {
  dsp_context* ctx = nullptr;
  int64_t n = 0, index_base = 0;
  int d = 0, dp = 0, k = 0;
  float tnorm_max = 0.f;
  // candidate scan, decided at fit: a train value outside the range of the tensor-core filter (knn_tc16.cu) / the dense
  // scan (knn_dense.cu) sends every call to the fp32 tiled / the float64 scan instead
  KnnScan scan = kScanF64;
  DevBuf tc_train, tc_train_rows, tc_q, tc_flags;      // train packed in tile order / in row order (knn_prune 0)
  DevBuf train64, train32, labels, tnorm, cand_idx, cand_worst, qnorm, redo_list, redo_count, nbr_label, q, o_idx, o_dist, o_lab;
  DevBuf refine_list, refine_thr, surv_count, surv_rows;     // second pass of the D <= 15 path (knn_refine)
  DevBuf thr0;                                               // bounded / pruned calls: per-query start thresholds of the filter
  DevBuf prune_perm, prune_geom, prune_box, prune_ws, prune_bound;   // tile pruning (knn_prune_plan / knn_prune_prepare)
  int64_t prune_tiles = 0;
  int refine_cap = 0;          // refine list capacity of the last call (rejected queries past it count in redo_count[1] too)
  DevBuf tpacked, tnorm_dense, qpacked, qnorm_chunk, dense_flags, part_d, part_i;
};

namespace {

int host_window(int type, int n, std::vector<double>& w) {
  if (n < 0) return fail(DSP_ERR_INVALID, "window length must be >= 0");
  w.assign((size_t)n, 1.0);
  if (type == DSP_WIN_RECTANGULAR) return DSP_OK;
  if (type != DSP_WIN_HAMMING && type != DSP_WIN_HANNING)
    return fail(DSP_ERR_INVALID, "unsupported window type: %d", type);   // audio_processing.py:296
  if (n <= 1) return DSP_OK;  // np.hamming(1) == np.hanning(1) == [1.]
  const double a = type == DSP_WIN_HAMMING ? 0.54 : 0.5, b = type == DSP_WIN_HAMMING ? 0.46 : 0.5;
  for (int i = 0; i < n; ++i) {
    const double m = (double)(1 - n + 2 * i);   // np: n = arange(1-M, M, 2)
    w[(size_t)i] = a + b * std::cos(M_PI * m / (double)(n - 1));
  }
  return DSP_OK;
}

int ensure_window(dsp_context* c, int type, int fl) {
  for (const auto& e : c->windows)
    if (e->type == type && e->len == fl) { c->win64 = e->w64.as<double>(); c->win32 = e->w32.as<float>(); return DSP_OK; }
  std::vector<double> w;
  int rc = host_window(type, fl, w);
  if (rc) return rc;
  std::vector<float> wf(w.begin(), w.end());
  if (c->windows.size() >= 256) {            // a pathological sweep: drop the tables once nothing can be reading them
    CU(cudaDeviceSynchronize());
    c->windows.clear();
  }
  auto e = std::make_unique<dsp_context::WinEntry>();
  e->type = type;
  e->len = fl;
  if (e->w64.ensure(sizeof(double) * (size_t)fl + 16) != cudaSuccess || e->w32.ensure(sizeof(float) * (size_t)fl + 16) != cudaSuccess)
    return fail(DSP_ERR_NOMEM, "device allocation failed");
  // a fresh table nobody reads yet: blocking copies from the stack vectors are safe and happen once per (type, length)
  CU(cudaMemcpy(e->w64.p, w.data(), sizeof(double) * (size_t)fl, cudaMemcpyHostToDevice));
  CU(cudaMemcpy(e->w32.p, wf.data(), sizeof(float) * (size_t)fl, cudaMemcpyHostToDevice));
  c->win64 = e->w64.as<double>(); c->win32 = e->w32.as<float>();
  c->windows.push_back(std::move(e));
  return DSP_OK;
}

int check_params(const dsp_frontend_params* p) {
  if (!p) return fail(DSP_ERR_INVALID, "params is NULL");
  if (p->frame_length < 1 || p->frame_shift < 1) return fail(DSP_ERR_INVALID, "frame_length and frame_shift must be >= 1");
  if (p->window < 0 || p->window > 2) return fail(DSP_ERR_INVALID, "unsupported window type: %d", p->window);
  if (p->channels != 1 && p->channels != 2) return fail(DSP_ERR_INVALID, "channels must be 1 or 2 (load_wav only down-mixes two channels, audio_processing.py:43-44: pass other files as 1 channel)");
  return DSP_OK;
}

struct ExactExtras {
  int pre_mode = 3, do_features = 1;
  double* pre_out = nullptr;
  double* frames_out = nullptr;
  double* epd_zcr_f64 = nullptr;
  double* feat_f64[3] = {nullptr, nullptr, nullptr};
  double* stats_f64 = nullptr;
};

int launch_exact(dsp_context* c, const void* samples, int dtype, const int64_t* offsets, const int32_t* lengths,
                 const int64_t* feat_offsets, const int64_t* epd_offsets, const int32_t* list,
                 const int32_t* list_count, int64_t n_items, int64_t max_len, const dsp_frontend_params* p,
                 const dsp_frontend_outputs* out, const ExactExtras& ex, int grid) {
  if (grid < 1) grid = 1;
  const int64_t cap_frames = std::max<int64_t>(frame_count_host_device(max_len, p->frame_length, p->frame_shift), 1);
  CU(c->zbuf.ensure(sizeof(double) * (size_t)grid * (size_t)std::max<int64_t>(max_len, 1)));
  CU(c->seqbuf.ensure(sizeof(double) * (size_t)grid * 5 * (size_t)cap_frames));
  ExactArgs a{};
  a.samples = samples; a.dtype = dtype; a.channels = p->channels;
  a.offsets = offsets; a.lengths = lengths; a.feat_offsets = feat_offsets; a.epd_offsets = epd_offsets;
  a.list = list; a.list_count = list_count; a.n_items = n_items;
  a.fl = p->frame_length; a.fs = p->frame_shift;
  a.do_epd = p->do_endpoint_detection; a.pre_mode = ex.pre_mode; a.do_features = ex.do_features;
  a.hr = p->energy_high_ratio; a.lr = p->energy_low_ratio; a.zr = p->zcr_threshold_ratio;
  a.win = c->win64;
  a.zbuf = c->zbuf.as<double>(); a.zbuf_stride = std::max<int64_t>(max_len, 1);
  a.seqbuf = c->seqbuf.as<double>(); a.seq_cap = cap_frames;
  if (out) a.out = *out;
  a.pre_out = ex.pre_out; a.frames_out = ex.frames_out; a.epd_zcr_f64 = ex.epd_zcr_f64;
  a.feat_f64[0] = ex.feat_f64[0]; a.feat_f64[1] = ex.feat_f64[1]; a.feat_f64[2] = ex.feat_f64[2];
  a.stats_f64 = ex.stats_f64;
  frontend_exact_kernel<<<grid, kExactThreads, 0, c->stream>>>(a);
  c->launches++;
  CU(cudaGetLastError());
  return DSP_OK;
}

// Kernel route of one front-end batch (DESIGN §3.1b), first match wins:
//   not int16 mono, force_exact, a float64 output, max_len > 2^20 or no feat_offsets  -> float64 replay
//   pcm_variant -1 or 10 and pipe_kernel_plan fits                                    -> frontend_pipe_kernel
//   pcm_variant 0..9                                                                  -> that frontend_pcm_kernel build
//   otherwise                                         -> build 2 (streaming) for aligned16 batches, else build 0 (resident)
//   the build fits no CTA on an SM (static + dynamic shared memory)                   -> float64 replay
// Alone, the replay runs on a grid of 4 x SMs and writes the float64 outputs; behind a fast kernel it runs on one CTA per
// SM and replays only the utterances that kernel flagged.
struct FrontRoute {
  enum Kind { kReplay, kPipe, kPcm } kind = kReplay;
  int build = 0;             // kPcm: index into frontend_pcm.cu's kVariants
  PipePlan plan{};           // kPipe
  int cap_samples = 0;       // kPcm
  size_t smem = 0;
  int grid = 0, replay_grid = 0;
};

FrontRoute route_frontend(dsp_context* c, int dtype, const int64_t* feat_offsets, int64_t B, int64_t max_len,
                          int cap_frames, const dsp_frontend_params* p, bool want64) {
  FrontRoute r;
  const int64_t sms = c->sm_count;
  r.replay_grid = (int)std::min<int64_t>(B, sms * 4);
  if (dtype != DSP_S16 || p->channels != 1 || p->force_exact || want64 || max_len > kFastMaxLen || !feat_offsets) return r;
  const int knob = c->pcm_variant, pipe_knob = pcm_num_variants();
  // the pipelined kernel first: 2.2-5x faster than build 0 on every geometry whose per-utterance records fit (DESIGN §3.1c)
  if ((knob < 0 || knob == pipe_knob) && pipe_kernel_plan(max_len, cap_frames, p->frame_length, kMaxSmemPerCta, &r.plan)) {
    r.kind = FrontRoute::kPipe;
    r.smem = r.plan.smem;
    r.grid = r.replay_grid = (int)std::min<int64_t>(B, sms);
    return r;
  }
  constexpr int kAutoStream = 2, kAutoResident = 0;
  r.build = knob >= 0 && knob < pipe_knob ? knob : (knob < 0 && p->aligned16 ? kAutoStream : kAutoResident);
  r.cap_samples = (int)((std::max<int64_t>(max_len, 1) + 63) / 64 * 64);
  r.smem = pcm_kernel_smem_bytes(r.cap_samples, cap_frames, p->frame_length, !pcm_variant_streams(r.build));
  if (c->occ_smem != r.smem || c->occ_variant != r.build) {
    c->occ = pcm_kernel_max_ctas_per_sm(r.build, r.smem, c->smem_optin);
    c->occ_smem = r.smem;
    c->occ_variant = r.build;
  }
  if (c->occ < 1) return r;
  r.kind = FrontRoute::kPcm;
  r.grid = (int)std::min<int64_t>(B, sms * c->occ);
  r.replay_grid = (int)std::min<int64_t>(B, sms);
  return r;
}

// DSP_PROF: per-phase cycle counters of the fast kernels, printed to stderr after every launch (tools/quick_pipe.py
// shows them).  Returns the zeroed counters, or nullptr when DSP_PROF is unset.
long long* prof_begin(dsp_context* c) {
  if (!std::getenv("DSP_PROF") || c->prof.ensure(16 * sizeof(long long)) != cudaSuccess) return nullptr;
  cudaMemsetAsync(c->prof.p, 0, 16 * sizeof(long long), c->stream);
  return c->prof.as<long long>();
}

void prof_report(dsp_context* c, const FrontRoute& r) {
  long long h[16];
  cudaMemcpyAsync(h, c->prof.p, sizeof h, cudaMemcpyDeviceToHost, c->stream);
  cudaStreamSynchronize(c->stream);
  if (r.kind == FrontRoute::kPipe) {
    const char* nm[12] = {"S.wait_full", "S.passA", "S.bar1", "S.passB", "S.bar2", "S.wait_rec", "S.passF", "-", "T.wait", "T.decide", "T.window", "T.stats+out"};
    // n_rec holds two batches of records, one per tail warp at work
    const int tail_warps = r.plan.n_rec / 2;
    fprintf(stderr, "[prof pipe R=%d nrec=%d] utterances=%lld (cycles/utt, stream warp 0 / tail warp 0 x %d tail warps)", r.plan.ring_slots, r.plan.n_rec, h[15], tail_warps);
    for (int i = 0; i < 12; ++i) fprintf(stderr, "  %s=%.0f", nm[i], (double)h[i] / (double)std::max<long long>(h[15], 1) * (i >= 8 ? tail_warps : 1));
    fprintf(stderr, "\n");
  } else {
    const char* nm[12] = {"load_wait", "P1", "feat_empty_wait", "P2", "P2b", "P3tail(searches)", "P4", "fixup+handoff", "P3a(select passes)", "P3b(gather)", "P3c(rank+thresholds)", "P3d(N3N4)"};
    double tot = 0; for (int i = 0; i < 12; ++i) tot += (double)h[i];
    fprintf(stderr, "[prof] utterances=%lld", h[15]); for (int i = 0; i < 12; ++i) fprintf(stderr, "  %s=%.0f", nm[i], (double)h[i] / (double)h[15]); fprintf(stderr, "  total=%.0f cycles/utt\n", tot / (double)h[15]);
  }
}

int frontend_device(dsp_context* c, const void* samples, int dtype, const int64_t* offsets, const int32_t* lengths,
                    const int64_t* feat_offsets, const int64_t* epd_offsets, int64_t B, int64_t max_len,
                    const dsp_frontend_params* p, const dsp_frontend_outputs* out) {
  int rc = check_params(p);
  if (rc) return rc;
  if (!dtype_size(dtype)) return fail(DSP_ERR_INVALID, "unsupported sample dtype %d", dtype);
  if (!out) return fail(DSP_ERR_INVALID, "outputs is NULL");
  if (B < 0 || max_len < 0) return fail(DSP_ERR_INVALID, "negative batch size or length");
  if (B == 0) return DSP_OK;
  if (B > INT32_MAX / 2) return fail(DSP_ERR_UNSUPPORTED, "more than 2^30 utterances in one call");
  if (p->channels == 2 && (dtype == DSP_F32 || dtype == DSP_F64))
    return fail(DSP_ERR_INVALID, "stereo input is only defined for PCM (load_wav)");
  if ((out->energy || out->magnitude || out->zcr) && !feat_offsets) return fail(DSP_ERR_INVALID, "feat_offsets is NULL");
  if ((out->epd_energy || out->epd_zcr) && !epd_offsets) return fail(DSP_ERR_INVALID, "epd_offsets is NULL");
  rc = ensure_window(c, p->window, p->frame_length);
  if (rc) return rc;
  const int cap_frames = (int)std::max<int64_t>(frame_count_host_device(max_len, p->frame_length, p->frame_shift), 1);

  const bool want64 = out->energy_f64 || out->magnitude_f64 || out->zcr_f64 || out->stats_f64 || out->epd_zcr_f64 || out->frames_f64;
  if (out->frames_f64 && !feat_offsets) return fail(DSP_ERR_INVALID, "feat_offsets is NULL");
  if ((out->energy_f64 || out->magnitude_f64 || out->zcr_f64) && !(out->energy_f64 && out->magnitude_f64 && out->zcr_f64))
    return fail(DSP_ERR_INVALID, "energy_f64, magnitude_f64 and zcr_f64 are written together: pass all three or none");
  if (out->energy_f64 && !feat_offsets) return fail(DSP_ERR_INVALID, "feat_offsets is NULL");
  if (out->epd_zcr_f64 && !epd_offsets) return fail(DSP_ERR_INVALID, "epd_offsets is NULL");
  const FrontRoute r = route_frontend(c, dtype, feat_offsets, B, max_len, cap_frames, p, want64);
  ExactExtras ex;
  PcmArgs a{};                // flag_list stays NULL on the replay route: the replay takes the whole batch
  if (r.kind == FrontRoute::kReplay) {
    ex.feat_f64[0] = out->energy_f64; ex.feat_f64[1] = out->magnitude_f64; ex.feat_f64[2] = out->zcr_f64;
    ex.stats_f64 = out->stats_f64; ex.epd_zcr_f64 = out->epd_zcr_f64; ex.frames_out = out->frames_f64;
  } else {
    CU(c->counters.ensure(64));
    CU(c->flag_list.ensure(sizeof(int32_t) * (size_t)B));
    CU(cudaMemsetAsync(c->counters.p, 0, 64, c->stream));
    a.samples = reinterpret_cast<const int16_t*>(samples);
    a.offsets = offsets; a.lengths = lengths; a.feat_offsets = feat_offsets; a.epd_offsets = epd_offsets;
    a.n_utts = B; a.fl = p->frame_length; a.fs = p->frame_shift; a.window = p->window; a.do_epd = p->do_endpoint_detection;
    a.hr = p->energy_high_ratio; a.lr = p->energy_low_ratio; a.zr = p->zcr_threshold_ratio;
    a.win_f32 = c->win32;
    a.cap_samples = r.cap_samples; a.cap_frames = cap_frames;
    a.tma_chunk = c->tma_chunk;
    a.stagger_ns = c->stagger_ns;
    a.sm_count = c->sm_count;
    a.ring_slots = r.plan.ring_slots; a.n_rec = r.plan.n_rec; a.cap_groups = r.plan.cap_groups;
    a.prof = prof_begin(c);
    a.work_counter = c->counters.as<unsigned int>();
    a.flag_count = c->counters.as<int32_t>() + 1;
    a.flag_list = c->flag_list.as<int32_t>();
    a.out = *out;
    if (r.kind == FrontRoute::kPipe) CU(launch_frontend_pipe(a, r.grid, r.smem, c->stream));
    else CU(launch_frontend_pcm(r.build, a, r.grid, r.smem, c->stream));
    if (a.prof) prof_report(c, r);
    c->launches++;
  }
  // behind a fast kernel: float64 replay of the utterances whose threshold margins could not be certified
  return launch_exact(c, samples, dtype, offsets, lengths, feat_offsets, epd_offsets, a.flag_list, a.flag_count,
                      a.flag_list ? 0 : B, max_len, p, out, ex, r.replay_grid);
}

int check_mfcc_params(const dsp_mfcc_params* p) {
  if (p->frame_length < 1 || p->frame_shift < 1 || p->n_mels < 1 || p->n_ceps < 1 || p->n_ceps > p->n_mels)
    return fail(DSP_ERR_INVALID, "bad MFCC geometry");
  if (p->n_fft < 32 || (p->n_fft & (p->n_fft - 1)) || p->n_fft < p->frame_length || p->n_fft > 16384)
    return fail(DSP_ERR_INVALID, "n_fft must be a power of two in [max(32, frame_length), 16384]");
  if (mfcc_smem_bytes(p->n_fft, p->n_mels) > kMaxSmemPerCta) return fail(DSP_ERR_UNSUPPORTED, "n_fft too large for shared memory");
  return DSP_OK;
}

// the tables mfcc_kernel reads besides the caller's filterbank / DCT: float32 window, twiddles, filter bin ranges
int mfcc_host_tables(const dsp_mfcc_params* p, const float* filterbank, std::vector<float>& wf, std::vector<float>& tw,
                     std::vector<int>& range) {
  std::vector<double> w;
  int rc = host_window(p->window, p->frame_length, w);
  if (rc) return rc;
  wf.assign(w.begin(), w.end());
  const int n_bins = p->n_fft / 2 + 1;
  tw.assign((size_t)p->n_fft, 0.f);                                               // W[k] = exp(-2 pi i k / n_fft), k < n_fft / 2
  for (int k = 0; k < p->n_fft / 2; ++k) {
    const double a = -2.0 * M_PI * (double)k / (double)p->n_fft;
    tw[2 * (size_t)k] = (float)std::cos(a); tw[2 * (size_t)k + 1] = (float)std::sin(a);
  }
  range.assign(2 * (size_t)p->n_mels, 0);                                         // non-zero bins of every filter
  for (int m = 0; m < p->n_mels; ++m) {
    int lo = n_bins, hi = 0;
    for (int b = 0; b < n_bins; ++b) if (filterbank[(size_t)m * n_bins + b] != 0.f) { lo = std::min(lo, b); hi = std::max(hi, b + 1); }
    range[2 * (size_t)m] = std::min(lo, hi); range[2 * (size_t)m + 1] = hi;
  }
  return DSP_OK;
}

// The context's device tables for these parameters and host tables, uploaded on first use (stream-ordered copies from
// host vectors the entry keeps).  A hit compares the tables on the host and copies nothing.
int ensure_mfcc_tables(dsp_context* c, const dsp_mfcc_params* p, const float* filterbank, const float* dct,
                       dsp_context::MfccEntry** out) {
  const size_t n_fb = (size_t)p->n_mels * (p->n_fft / 2 + 1), n_dct = (size_t)p->n_ceps * p->n_mels;
  for (const auto& e : c->mfcc_tables)
    if (e->frame_length == p->frame_length && e->window == p->window && e->n_fft == p->n_fft && e->n_mels == p->n_mels &&
        e->n_ceps == p->n_ceps && !std::memcmp(e->fb.data(), filterbank, n_fb * sizeof(float)) &&
        !std::memcmp(e->dct.data(), dct, n_dct * sizeof(float))) { *out = e.get(); return DSP_OK; }
  if (c->mfcc_tables.size() >= 16) {           // a sweep over many geometries: drop the tables once nothing can be reading them
    CU(cudaDeviceSynchronize());
    c->mfcc_tables.clear();
  }
  auto e = std::make_unique<dsp_context::MfccEntry>();
  e->frame_length = p->frame_length;
  e->window = p->window;
  e->n_fft = p->n_fft;
  e->n_mels = p->n_mels;
  e->n_ceps = p->n_ceps;
  e->fb.assign(filterbank, filterbank + n_fb);
  e->dct.assign(dct, dct + n_dct);
  int rc = mfcc_host_tables(p, filterbank, e->win, e->tw, e->range);
  if (rc) return rc;
  if (e->d_win.ensure(sizeof(float) * e->win.size()) != cudaSuccess || e->d_tw.ensure(sizeof(float) * e->tw.size()) != cudaSuccess ||
      e->d_fb.ensure(sizeof(float) * n_fb) != cudaSuccess || e->d_range.ensure(sizeof(int) * e->range.size()) != cudaSuccess ||
      e->d_dct.ensure(sizeof(float) * n_dct) != cudaSuccess)
    return fail(DSP_ERR_NOMEM, "device allocation failed");
  CU(cudaMemcpyAsync(e->d_win.p, e->win.data(), sizeof(float) * e->win.size(), cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(e->d_tw.p, e->tw.data(), sizeof(float) * e->tw.size(), cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(e->d_fb.p, e->fb.data(), sizeof(float) * n_fb, cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(e->d_range.p, e->range.data(), sizeof(int) * e->range.size(), cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(e->d_dct.p, e->dct.data(), sizeof(float) * n_dct, cudaMemcpyHostToDevice, c->stream));
  *out = e.get();
  c->mfcc_tables.push_back(std::move(e));
  return DSP_OK;
}

// small helper for the single-signal host entry points: scratch buffers from the context, nullptr past the last one
struct OneShot {
  dsp_context* c;
  int n_tmp = 0;
  explicit OneShot(dsp_context* ctx) : c(ctx) {}
  template <class T> T* dev(size_t count) {
    if (n_tmp == (int)std::size(c->tmp)) return nullptr;
    DevBuf& b = c->tmp[n_tmp++];
    if (b.ensure(sizeof(T) * std::max<size_t>(count, 1)) != cudaSuccess) return nullptr;
    return b.as<T>();
  }
};

}  // namespace

// =============================================================================================
extern "C" {

int dsp_abi_version(void) { return DSPFRONT_ABI_VERSION; }
const char* dsp_last_error(void) { return g_err.c_str(); }

int dsp_create(int device, dsp_context** out) {
  if (!out) return fail(DSP_ERR_INVALID, "out is NULL");
  *out = nullptr;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) {
    cudaGetLastError();
    return fail(DSP_ERR_NO_DEVICE, "no CUDA device: libdspfront has no CPU path");
  }
  if (device < 0 || device >= count) return fail(DSP_ERR_INVALID, "device %d out of range (%d visible)", device, count);
  CU(cudaSetDevice(device));
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) return fail(DSP_ERR_NO_DEVICE, "device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
  auto c = std::make_unique<dsp_context>();
  c->device = device;
  c->sm_count = prop.multiProcessorCount;
  c->smem_optin = prop.sharedMemPerBlockOptin;
  CU(cudaStreamCreateWithFlags(&c->own.h, cudaStreamNonBlocking));
  CU(cudaStreamCreateWithFlags(&c->s_in.h, cudaStreamNonBlocking));
  CU(cudaStreamCreateWithFlags(&c->s_out.h, cudaStreamNonBlocking));
  c->stream = c->own;
  if (const char* e = std::getenv("DSP_PCM_VARIANT")) { int v = std::atoi(e); if (v >= -1 && v <= pcm_num_variants()) c->pcm_variant = v; }
  if (const char* e = std::getenv("DSP_STAGGER_NS")) c->stagger_ns = std::atoi(e);
  if (const char* e = std::getenv("DSP_TMA_CHUNK")) { int v = std::atoi(e); if (v >= 16 && v % 16 == 0) c->tma_chunk = v; }
  for (auto& s : c->slot) {
    CU(cudaEventCreateWithFlags(&s.ev_in.h, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&s.ev_k.h, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&s.ev_out.h, cudaEventDisableTiming));
  }
  *out = c.release();
  return DSP_OK;
}

int dsp_destroy(dsp_context* c) {
  if (!c) return DSP_OK;
  const std::unique_ptr<dsp_context> owner(c);   // its members free the buffers, tables, events and streams
  cudaSetDevice(c->device);
  cudaDeviceSynchronize();
  return DSP_OK;
}

int dsp_set_stream(dsp_context* c, void* cuda_stream) {
  if (!c) return fail(DSP_ERR_INVALID, "context is NULL");
  c->stream = reinterpret_cast<cudaStream_t>(cuda_stream);
  return DSP_OK;
}

int dsp_use_own_stream(dsp_context* c) {
  if (!c) return fail(DSP_ERR_INVALID, "context is NULL");
  c->stream = c->own;
  return DSP_OK;
}

int dsp_set_tuning(dsp_context* c, const char* key, int value) {
  if (!c || !key) return fail(DSP_ERR_INVALID, "bad argument");
  if (!std::strcmp(key, "pcm_variant")) {
    if (value < -1 || value > pcm_num_variants()) return fail(DSP_ERR_INVALID, "pcm_variant out of range (%d builds + the pipelined kernel)", pcm_num_variants());
    c->pcm_variant = value;
  } else if (!std::strcmp(key, "tma_chunk")) {
    if (value < 16 || value % 16) return fail(DSP_ERR_INVALID, "tma_chunk must be a positive multiple of 16");
    c->tma_chunk = value;
  } else if (!std::strcmp(key, "stagger_ns")) {
    c->stagger_ns = value;
  } else if (!std::strcmp(key, "knn_prune")) {
    if (value < 0 || value > 2) return fail(DSP_ERR_INVALID, "knn_prune must be 0 (off), 1 (automatic) or 2 (always)");
    c->knn_prune = value;
  } else {
    return fail(DSP_ERR_INVALID, "unknown tuning key '%s'", key);
  }
  return DSP_OK;
}

int dsp_sync(dsp_context* c) {
  if (!c) return fail(DSP_ERR_INVALID, "context is NULL");
  CU(cudaSetDevice(c->device));
  CU(cudaStreamSynchronize(c->stream));
  return DSP_OK;
}

int64_t dsp_launch_count(dsp_context* c) { return c ? c->launches : 0; }
int dsp_device_sm_count(dsp_context* c) { return c ? c->sm_count : 0; }

int64_t dsp_frame_count(int64_t n, int32_t fl, int32_t fs) {
  if (fl < 1 || fs < 1) return 0;
  return frame_count_host_device(n, fl, fs);
}

int dsp_frontend_plan(const int64_t* offsets, const int32_t* lengths, int64_t B, const dsp_frontend_params* p,
                      int64_t* feat_offsets, int64_t* epd_offsets, int64_t* max_len) {
  int rc = check_params(p);
  if (rc) return rc;
  if (!offsets || B < 0) return fail(DSP_ERR_INVALID, "bad offsets");
  int64_t fo = 0, eo = 0, mx = 0;
  for (int64_t b = 0; b < B; ++b) {
    const int64_t room = offsets[b + 1] - offsets[b];
    const int64_t len = lengths ? (int64_t)lengths[b] : room;
    if (room < 0 || len < 0 || len > room || len % p->channels)
      return fail(DSP_ERR_INVALID, "offsets must be non-decreasing, lengths must fit and be a multiple of channels (utterance %lld)", (long long)b);
    const int64_t n = len / p->channels;
    if (n > INT32_MAX / 4) return fail(DSP_ERR_UNSUPPORTED, "utterance %lld is too long", (long long)b);
    if (feat_offsets) feat_offsets[b] = fo;
    if (epd_offsets) epd_offsets[b] = eo;
    fo += frame_count_host_device(n, p->frame_length, p->frame_shift);
    eo += (p->do_endpoint_detection && n >= p->frame_length) ? (n - p->frame_length) / p->frame_shift + 1 : 0;
    mx = std::max(mx, n);
  }
  if (feat_offsets) feat_offsets[B] = fo;
  if (epd_offsets) epd_offsets[B] = eo;
  if (max_len) *max_len = mx;
  return DSP_OK;
}

int dsp_window(int window_type, int32_t length, double* out) {
  std::vector<double> w;
  int rc = host_window(window_type, length, w);
  if (rc) return rc;
  if (length > 0 && !out) return fail(DSP_ERR_INVALID, "out is NULL");
  std::memcpy(out, w.data(), sizeof(double) * w.size());
  return DSP_OK;
}

int dsp_frontend_batch_device(dsp_context* c, const void* samples, int dtype, const int64_t* offsets,
                              const int32_t* lengths, const int64_t* feat_offsets, const int64_t* epd_offsets, int64_t n_utts,
                              int64_t max_len, const dsp_frontend_params* p, const dsp_frontend_outputs* out) {
  if (!c) return fail(DSP_ERR_INVALID, "context is NULL");
  CU(cudaSetDevice(c->device));
  return frontend_device(c, samples, dtype, offsets, lengths, feat_offsets, epd_offsets, n_utts, max_len, p, out);
}

int dsp_frontend_batch_host(dsp_context* c, const void* samples, int dtype, const int64_t* offsets,
                            const int32_t* lengths, int64_t B, const dsp_frontend_params* p, const dsp_frontend_outputs* out) {
  if (!c) return fail(DSP_ERR_INVALID, "context is NULL");
  int rc = check_params(p);
  if (rc) return rc;
  const size_t esz = dtype_size(dtype);
  if (!esz) return fail(DSP_ERR_INVALID, "unsupported sample dtype %d", dtype);
  if (!out || !offsets) return fail(DSP_ERR_INVALID, "NULL argument");
  if (B == 0) return DSP_OK;
  CU(cudaSetDevice(c->device));
  std::vector<int64_t> foff((size_t)B + 1), eoff((size_t)B + 1);
  int64_t max_len_all = 0;
  rc = dsp_frontend_plan(offsets, lengths, B, p, foff.data(), eoff.data(), &max_len_all);
  if (rc) return rc;
  rc = ensure_window(c, p->window, p->frame_length);
  if (rc) return rc;

  // every return, an error inside the chunk loop included, waits until no download into the caller's arrays is in flight
  struct DrainDownloads {
    cudaStream_t s_out;
    ~DrainDownloads() { cudaStreamSynchronize(s_out); }
  } drain_on_return{c->s_out};
  const unsigned char* src = reinterpret_cast<const unsigned char*>(samples);
  int64_t b0 = 0;
  int chunk = 0;
  while (b0 < B) {
    // chunk = as many utterances as fit the staging budget (at least one)
    int64_t b1 = b0 + 1;
    while (b1 < B && (size_t)(offsets[b1 + 1] - offsets[b0]) * esz <= host_chunk_bytes()) ++b1;
    const int64_t bc = b1 - b0;
    Slot& s = c->slot[chunk & 1];
    if (chunk >= 2) CU(cudaEventSynchronize(s.ev_out));   // the downloads of chunk - 2 read this slot's buffers
    const int64_t e0 = offsets[b0], e1 = offsets[b1];
    const int64_t f0 = foff[(size_t)b0], f1 = foff[(size_t)b1], g0 = eoff[(size_t)b0], g1 = eoff[(size_t)b1];
    CU(s.h_off.ensure(sizeof(int64_t) * 4 * (size_t)(bc + 1)));
    int64_t* h = s.h_off.as<int64_t>();
    int64_t chunk_max = 0;
    for (int64_t i = 0; i <= bc; ++i) {
      h[i] = offsets[b0 + i] - e0;
      h[(bc + 1) + i] = foff[(size_t)(b0 + i)] - f0;
      h[2 * (bc + 1) + i] = eoff[(size_t)(b0 + i)] - g0;
      if (i < bc) {
        const int64_t len = lengths ? (int64_t)lengths[b0 + i] : offsets[b0 + i + 1] - offsets[b0 + i];
        chunk_max = std::max(chunk_max, len / p->channels);
        reinterpret_cast<int32_t*>(h + 3 * (bc + 1))[i] = (int32_t)len;
      }
    }
    CU(s.samples.ensure((size_t)(e1 - e0) * esz + 64));
    CU(s.off.ensure(sizeof(int64_t) * 4 * (size_t)(bc + 1)));
    CU(s.ints.ensure(sizeof(int32_t) * 5 * (size_t)bc));
    CU(s.stats.ensure(sizeof(float) * kStats * (size_t)bc));
    CU(s.feat.ensure(sizeof(float) * 3 * (size_t)std::max<int64_t>(f1 - f0, 1)));
    CU(s.epd_e.ensure(sizeof(double) * (size_t)std::max<int64_t>(g1 - g0, 1)));
    CU(s.epd_z.ensure(sizeof(float) * (size_t)std::max<int64_t>(g1 - g0, 1)));
    const bool want64 = out->energy_f64 || out->magnitude_f64 || out->zcr_f64 || out->stats_f64 || out->epd_zcr_f64 || out->frames_f64;
    const int64_t fn64 = std::max<int64_t>(f1 - f0, 1), gn64 = std::max<int64_t>(g1 - g0, 1);
    const size_t dense64 = out->frames_f64 ? (size_t)fn64 * (size_t)p->frame_length : 0;
    if (want64) CU(s.f64.ensure(sizeof(double) * ((size_t)(3 * fn64 + kStats * bc + gn64) + dense64)));
    // upload
    CU(cudaMemcpyAsync(s.samples.p, src + (size_t)e0 * esz, (size_t)(e1 - e0) * esz, cudaMemcpyHostToDevice, c->s_in));
    CU(cudaMemcpyAsync(s.off.p, h, sizeof(int64_t) * 4 * (size_t)(bc + 1), cudaMemcpyHostToDevice, c->s_in));
    CU(cudaEventRecord(s.ev_in, c->s_in));
    CU(cudaStreamWaitEvent(c->stream, s.ev_in, 0));
    // kernels
    int32_t* di = s.ints.as<int32_t>();
    float* df = s.feat.as<float>();
    const int64_t fn = std::max<int64_t>(f1 - f0, 1);
    dsp_frontend_outputs o{};
    o.start = di; o.end = di + bc; o.n_epd_frames = di + 2 * bc; o.n_frames = di + 3 * bc; o.status = di + 4 * bc;
    o.energy = df; o.magnitude = df + fn; o.zcr = df + 2 * fn;
    o.stats = s.stats.as<float>();
    o.epd_energy = out->epd_energy ? s.epd_e.as<double>() : nullptr;
    o.epd_zcr = out->epd_zcr ? s.epd_z.as<float>() : nullptr;
    if (want64) {
      double* d64 = s.f64.as<double>();
      if (out->energy_f64) { o.energy_f64 = d64; o.magnitude_f64 = d64 + fn64; o.zcr_f64 = d64 + 2 * fn64; }
      if (out->stats_f64) o.stats_f64 = d64 + 3 * fn64;
      if (out->epd_zcr_f64) o.epd_zcr_f64 = d64 + 3 * fn64 + kStats * bc;
      if (out->frames_f64) o.frames_f64 = d64 + 3 * fn64 + kStats * bc + gn64;
    }
    const int64_t* doff = s.off.as<int64_t>();
    dsp_frontend_params pc = *p;
    pc.aligned16 = 1;                               // staging buffers come from cudaMalloc (256-byte aligned)
    for (int64_t i = 0; i < bc && pc.aligned16; ++i) if ((size_t)h[i] * esz % 16) pc.aligned16 = 0;
    const int32_t* dlen = lengths ? reinterpret_cast<const int32_t*>(doff + 3 * (bc + 1)) : nullptr;
    rc = frontend_device(c, s.samples.p, dtype, doff, dlen, doff + (bc + 1), doff + 2 * (bc + 1), bc, chunk_max, &pc, &o);
    if (rc) return rc;
    CU(cudaEventRecord(s.ev_k, c->stream));
    CU(cudaStreamWaitEvent(c->s_out, s.ev_k, 0));
    // download straight into the caller's arrays
    auto d2h = [&](void* dst, const void* srcp, size_t bytes) -> cudaError_t {
      if (!dst || bytes == 0) return cudaSuccess;
      return cudaMemcpyAsync(dst, srcp, bytes, cudaMemcpyDeviceToHost, c->s_out);
    };
    CU(d2h(out->start ? out->start + b0 : nullptr, o.start, sizeof(int32_t) * (size_t)bc));
    CU(d2h(out->end ? out->end + b0 : nullptr, o.end, sizeof(int32_t) * (size_t)bc));
    CU(d2h(out->n_epd_frames ? out->n_epd_frames + b0 : nullptr, o.n_epd_frames, sizeof(int32_t) * (size_t)bc));
    CU(d2h(out->n_frames ? out->n_frames + b0 : nullptr, o.n_frames, sizeof(int32_t) * (size_t)bc));
    CU(d2h(out->status ? out->status + b0 : nullptr, o.status, sizeof(int32_t) * (size_t)bc));
    CU(d2h(out->stats ? out->stats + b0 * kStats : nullptr, o.stats, sizeof(float) * kStats * (size_t)bc));
    CU(d2h(out->energy ? out->energy + f0 : nullptr, o.energy, sizeof(float) * (size_t)(f1 - f0)));
    CU(d2h(out->magnitude ? out->magnitude + f0 : nullptr, o.magnitude, sizeof(float) * (size_t)(f1 - f0)));
    CU(d2h(out->zcr ? out->zcr + f0 : nullptr, o.zcr, sizeof(float) * (size_t)(f1 - f0)));
    CU(d2h(out->epd_energy ? out->epd_energy + g0 : nullptr, o.epd_energy, sizeof(double) * (size_t)(g1 - g0)));
    CU(d2h(out->epd_zcr ? out->epd_zcr + g0 : nullptr, o.epd_zcr, sizeof(float) * (size_t)(g1 - g0)));
    CU(d2h(out->energy_f64 ? out->energy_f64 + f0 : nullptr, o.energy_f64, sizeof(double) * (size_t)(f1 - f0)));
    CU(d2h(out->magnitude_f64 ? out->magnitude_f64 + f0 : nullptr, o.magnitude_f64, sizeof(double) * (size_t)(f1 - f0)));
    CU(d2h(out->zcr_f64 ? out->zcr_f64 + f0 : nullptr, o.zcr_f64, sizeof(double) * (size_t)(f1 - f0)));
    CU(d2h(out->stats_f64 ? out->stats_f64 + b0 * kStats : nullptr, o.stats_f64, sizeof(double) * kStats * (size_t)bc));
    CU(d2h(out->epd_zcr_f64 ? out->epd_zcr_f64 + g0 : nullptr, o.epd_zcr_f64, sizeof(double) * (size_t)(g1 - g0)));
    CU(d2h(out->frames_f64 ? out->frames_f64 + (size_t)f0 * (size_t)p->frame_length : nullptr, o.frames_f64, sizeof(double) * (size_t)(f1 - f0) * (size_t)p->frame_length));
    CU(cudaEventRecord(s.ev_out, c->s_out));
    b0 = b1;
    ++chunk;
  }
  CU(cudaStreamSynchronize(c->s_out));
  return DSP_OK;
}

// ---- single-signal entry points (the per-call Python surface) -------------------------------
static int one_signal(dsp_context* c, const double* x, int64_t n, const dsp_frontend_params* p,
                      const ExactExtras& ex_in, dsp_frontend_outputs* dout, OneShot& os) {
  int rc = ensure_window(c, p->window, p->frame_length);
  if (rc) return rc;
  double* dx = os.dev<double>((size_t)n);
  int64_t* doff = os.dev<int64_t>(2);
  if (!dx || !doff) return fail(DSP_ERR_NOMEM, "device allocation failed");
  const int64_t hoff[2] = {0, n};
  CU(cudaMemcpyAsync(dx, x, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(doff, hoff, sizeof hoff, cudaMemcpyHostToDevice, c->stream));
  CU(cudaStreamSynchronize(c->stream));  // hoff is a stack array
  return launch_exact(c, dx, DSP_F64, doff, nullptr, nullptr, nullptr, nullptr, nullptr, 1, n, p, dout, ex_in, 1);
}

int dsp_preprocess_host(dsp_context* c, const double* x, int64_t n, int mode, double* out) {
  if (!c || (!x && n) || (!out && n) || n < 0 || mode < 0 || mode > 2) return fail(DSP_ERR_INVALID, "bad argument");
  if (n == 0) return fail(DSP_ERR_INVALID, "zero-size array to reduction operation maximum which has no identity");
  CU(cudaSetDevice(c->device));
  dsp_frontend_params p{};
  p.frame_length = 1; p.frame_shift = 1; p.window = 0; p.channels = 1;
  OneShot os(c);
  double* dout = os.dev<double>((size_t)n);
  if (!dout) return fail(DSP_ERR_NOMEM, "device allocation failed");
  ExactExtras ex;
  ex.pre_mode = mode == 0 ? 1 : (mode == 1 ? 2 : 3);
  ex.do_features = 0;
  ex.pre_out = dout;
  dsp_frontend_outputs o{};
  int rc = one_signal(c, x, n, &p, ex, &o, os);
  if (rc) return rc;
  CU(cudaMemcpyAsync(out, dout, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return DSP_OK;
}

int dsp_endpoint_detection_host(dsp_context* c, const double* x, int64_t n, const dsp_frontend_params* p,
                                int32_t* start, int32_t* end, int32_t* n_epd_frames, double* energy_list,
                                double* zcr_list) {
  if (!c || (!x && n) || n < 0) return fail(DSP_ERR_INVALID, "bad argument");
  int rc = check_params(p);
  if (rc) return rc;
  CU(cudaSetDevice(c->device));
  dsp_frontend_params q = *p;
  q.do_endpoint_detection = 1; q.channels = 1; q.window = DSP_WIN_RECTANGULAR;
  const int64_t f1 = n >= q.frame_length ? (n - q.frame_length) / q.frame_shift + 1 : 0;
  OneShot os(c);
  int32_t* di = os.dev<int32_t>(8);
  double* de = os.dev<double>((size_t)f1);
  double* dz = os.dev<double>((size_t)f1);
  if (!di || !de || !dz) return fail(DSP_ERR_NOMEM, "device allocation failed");
  ExactExtras ex;
  ex.pre_mode = 0; ex.do_features = 0; ex.epd_zcr_f64 = dz;
  dsp_frontend_outputs o{};
  o.start = di; o.end = di + 1; o.n_epd_frames = di + 2; o.epd_energy = de;
  // one_signal passes epd_offsets == NULL -> offset 0
  rc = one_signal(c, x, n, &q, ex, &o, os);
  if (rc) return rc;
  int32_t hi[3];
  CU(cudaMemcpyAsync(hi, di, sizeof hi, cudaMemcpyDeviceToHost, c->stream));
  if (energy_list && f1) CU(cudaMemcpyAsync(energy_list, de, sizeof(double) * (size_t)f1, cudaMemcpyDeviceToHost, c->stream));
  if (zcr_list && f1) CU(cudaMemcpyAsync(zcr_list, dz, sizeof(double) * (size_t)f1, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  if (start) *start = hi[0];
  if (end) *end = hi[1];
  if (n_epd_frames) *n_epd_frames = hi[2];
  return DSP_OK;
}

int dsp_frame_signal_host(dsp_context* c, const double* x, int64_t n, int32_t fl, int32_t fs, int window_type,
                          double* frames_out) {
  if (!c || (!x && n) || n < 0) return fail(DSP_ERR_INVALID, "bad argument");
  dsp_frontend_params p{};
  p.frame_length = fl; p.frame_shift = fs; p.window = window_type; p.channels = 1;
  int rc = check_params(&p);
  if (rc) return rc;
  const int64_t nf = frame_count_host_device(n, fl, fs);
  if (nf == 0) return DSP_OK;
  if (!frames_out) return fail(DSP_ERR_INVALID, "frames_out is NULL");
  CU(cudaSetDevice(c->device));
  OneShot os(c);
  double* dfr = os.dev<double>((size_t)nf * (size_t)fl);
  if (!dfr) return fail(DSP_ERR_NOMEM, "device allocation failed");
  ExactExtras ex;
  ex.pre_mode = 0; ex.do_features = 1; ex.frames_out = dfr;
  dsp_frontend_outputs o{};
  rc = one_signal(c, x, n, &p, ex, &o, os);
  if (rc) return rc;
  CU(cudaMemcpyAsync(frames_out, dfr, sizeof(double) * (size_t)nf * (size_t)fl, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return DSP_OK;
}

int dsp_frame_features_host(dsp_context* c, const double* frames, int64_t n_frames, int32_t fl, double* energy,
                            double* magnitude, double* zcr, double* stats) {
  if (!c || n_frames < 0 || fl < 0) return fail(DSP_ERR_INVALID, "bad argument");
  if (n_frames == 0) return fail(DSP_ERR_INVALID, "No frames provided for feature extraction.");  // feature_extraction.py:27-28
  if (n_frames > INT32_MAX) return fail(DSP_ERR_UNSUPPORTED, "too many frames");
  CU(cudaSetDevice(c->device));
  OneShot os(c);
  double* dfr = os.dev<double>((size_t)n_frames * (size_t)fl);
  double* de = os.dev<double>((size_t)n_frames * 3);
  double* dst = os.dev<double>(kStats);
  if (!dfr || !de || !dst) return fail(DSP_ERR_NOMEM, "device allocation failed");
  double* dm = de + n_frames; double* dz = dm + n_frames;
  if (fl > 0) CU(cudaMemcpyAsync(dfr, frames, sizeof(double) * (size_t)n_frames * (size_t)fl, cudaMemcpyHostToDevice, c->stream));
  frame_features_kernel<<<(unsigned)((n_frames + 127) / 128), 128, 0, c->stream>>>(dfr, n_frames, fl, de, dm, dz);
  c->launches++;
  CU(cudaGetLastError());
  if (stats) {
    sequence_stats_kernel<<<1, kExactThreads, 0, c->stream>>>(de, dm, dz, (int)n_frames, dst);
    c->launches++;
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(stats, dst, sizeof(double) * kStats, cudaMemcpyDeviceToHost, c->stream));
  }
  if (energy) CU(cudaMemcpyAsync(energy, de, sizeof(double) * (size_t)n_frames, cudaMemcpyDeviceToHost, c->stream));
  if (magnitude) CU(cudaMemcpyAsync(magnitude, dm, sizeof(double) * (size_t)n_frames, cudaMemcpyDeviceToHost, c->stream));
  if (zcr) CU(cudaMemcpyAsync(zcr, dz, sizeof(double) * (size_t)n_frames, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return DSP_OK;
}

int dsp_sequence_stats_host(dsp_context* c, const double* seq, int64_t n, double* out5) {
  if (!c || !out5 || n < 0) return fail(DSP_ERR_INVALID, "bad argument");
  if (n == 0) return fail(DSP_ERR_INVALID, "zero-size array to reduction operation maximum which has no identity");
  if (n > INT32_MAX) return fail(DSP_ERR_UNSUPPORTED, "sequence too long");
  CU(cudaSetDevice(c->device));
  OneShot os(c);
  double* ds = os.dev<double>((size_t)n);
  double* dst = os.dev<double>(kStats);
  if (!ds || !dst) return fail(DSP_ERR_NOMEM, "device allocation failed");
  CU(cudaMemcpyAsync(ds, seq, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, c->stream));
  sequence_stats_kernel<<<1, kExactThreads, 0, c->stream>>>(ds, nullptr, nullptr, (int)n, dst);
  c->launches++;
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(out5, dst, sizeof(double) * 5, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return DSP_OK;
}

int dsp_zscore_device(dsp_context* c, const double* x, int64_t n, int32_t d, int fit, double* mean, double* std,
                      double* out) {
  if (!c || n < 0 || d < 1 || !mean || !std) return fail(DSP_ERR_INVALID, "bad argument");
  CU(cudaSetDevice(c->device));
  if (fit) {
    if (n == 0) return fail(DSP_ERR_INVALID, "cannot fit on zero rows");
    CU(zscore_fit(x, n, d, (fit == 2) ? 1 : 0, mean, std, c->stream));
    c->launches++;
  }
  if (out) { CU(zscore_apply(x, n, d, mean, std, out, c->stream)); c->launches += 2; }
  return DSP_OK;
}

int dsp_zscore_apply_f32_device(dsp_context* c, const float* x, int64_t n, int32_t d, const double* mean,
                                const double* std, double* out) {
  if (!c || n < 0 || d < 1 || !mean || !std || (n && (!x || !out))) return fail(DSP_ERR_INVALID, "bad argument");
  CU(cudaSetDevice(c->device));
  CU(zscore_apply_f32(x, n, d, mean, std, out, c->stream));
  c->launches++;
  return DSP_OK;
}

int dsp_zscore_host(dsp_context* c, const double* x, int64_t n, int32_t d, int fit, double* mean, double* std,
                    double* out) {
  if (!c || n < 0 || d < 1 || !mean || !std || (!x && n)) return fail(DSP_ERR_INVALID, "bad argument");
  CU(cudaSetDevice(c->device));
  OneShot os(c);
  double* dx = os.dev<double>((size_t)n * d);
  double* dm = os.dev<double>((size_t)d);
  double* ds = os.dev<double>((size_t)d);
  double* dy = os.dev<double>((size_t)n * d);
  if (!dx || !dm || !ds || !dy) return fail(DSP_ERR_NOMEM, "device allocation failed");
  CU(cudaMemcpyAsync(dx, x, sizeof(double) * (size_t)n * d, cudaMemcpyHostToDevice, c->stream));
  if (!fit) {
    CU(cudaMemcpyAsync(dm, mean, sizeof(double) * d, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(ds, std, sizeof(double) * d, cudaMemcpyHostToDevice, c->stream));
  }
  int rc = dsp_zscore_device(c, dx, n, d, fit, dm, ds, out ? dy : nullptr);
  if (rc) return rc;
  CU(cudaMemcpyAsync(mean, dm, sizeof(double) * d, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaMemcpyAsync(std, ds, sizeof(double) * d, cudaMemcpyDeviceToHost, c->stream));
  if (out) CU(cudaMemcpyAsync(out, dy, sizeof(double) * (size_t)n * d, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return DSP_OK;
}

// ---- KNN ----------------------------------------------------------------------------------------
int dsp_knn_fit_device(dsp_context* c, const double* train, const int32_t* labels, int64_t n, int32_t d, int32_t k,
                       int64_t index_base, dsp_knn** out) {
  if (!c || !out || n < 1 || d < 1 || k < 1 || !train || !labels) return fail(DSP_ERR_INVALID, "bad argument");
  if (k > kKnnMaxK) return fail(DSP_ERR_UNSUPPORTED, "n_neighbors > %d is not supported", kKnnMaxK);
  if (n > INT32_MAX) return fail(DSP_ERR_UNSUPPORTED, "more than 2^31 train rows per shard");
  CU(cudaSetDevice(c->device));
  auto h = std::make_unique<dsp_knn>();
  h->ctx = c; h->n = n; h->d = d; h->k = k; h->index_base = index_base; h->dp = knn_padded_dim(d);
  if (h->train64.ensure(sizeof(double) * (size_t)n * d) != cudaSuccess || h->labels.ensure(sizeof(int32_t) * (size_t)n) != cudaSuccess ||
      h->tnorm.ensure(64) != cudaSuccess || h->redo_count.ensure(64) != cudaSuccess)
    return fail(DSP_ERR_NOMEM, "device allocation failed");
  CU(cudaMemcpyAsync(h->train64.p, train, sizeof(double) * (size_t)n * d, cudaMemcpyDeviceToDevice, c->stream));
  CU(cudaMemcpyAsync(h->labels.p, labels, sizeof(int32_t) * (size_t)n, cudaMemcpyDeviceToDevice, c->stream));
  if (h->dp) {
    if (h->train32.ensure(sizeof(float) * (size_t)n * h->dp) != cudaSuccess) return fail(DSP_ERR_NOMEM, "device allocation failed");
    CU(knn_pack(h->train64.as<double>(), n, d, h->dp, h->train32.as<float>(), h->tnorm.as<float>(), c->stream));
    c->launches++;
    CU(cudaMemcpyAsync(&h->tnorm_max, h->tnorm.p, sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  }
  int tc_flags[2] = {0, 1};
  if (h->dp == 16 && n >= 64 && k < kKnnCand && std::getenv("DSP_KNN_NO_TC16") == nullptr) {
    // the 15-dim statistical features: split-fp16 operands in tensor-core tile order, |t|^2 as the 16th feature; tc_train
    // holds the rows in the tile order of the pruning plan (principal-axis median splits), train64 / train32 keep the
    // original order
    std::vector<double> host((size_t)n * d);
    CU(cudaMemcpyAsync(host.data(), h->train64.p, sizeof(double) * host.size(), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    KnnPrunePlan plan;
    knn_prune_plan(host.data(), n, d, plan);
    h->prune_tiles = (int64_t)plan.slack.size();
    const size_t box = sizeof(double) * plan.lo.size();
    if (h->tc_train.ensure(knn_tc16_packed_bytes(n, false)) != cudaSuccess || h->tc_flags.ensure(64) != cudaSuccess ||
        h->prune_perm.ensure(sizeof(int) * (size_t)n) != cudaSuccess || h->prune_geom.ensure(sizeof(KnnPruneGeom)) != cudaSuccess ||
        h->prune_box.ensure(2 * box + sizeof(double) * plan.slack.size()) != cudaSuccess)
      return fail(DSP_ERR_NOMEM, "device allocation failed");
    unsigned char* pb = h->prune_box.as<unsigned char>();
    CU(cudaMemcpyAsync(h->prune_perm.p, plan.perm.data(), sizeof(int) * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(h->prune_geom.p, &plan.geom, sizeof(KnnPruneGeom), cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(pb, plan.lo.data(), box, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(pb + box, plan.hi.data(), box, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(pb + 2 * box, plan.slack.data(), sizeof(double) * plan.slack.size(), cudaMemcpyHostToDevice, c->stream));
    if (h->tc_train_rows.ensure(knn_tc16_packed_bytes(n, false)) != cudaSuccess) return fail(DSP_ERR_NOMEM, "device allocation failed");
    // row order for unpruned calls: a walk over spatially ordered tiles finds its neighbours late, and the filter pays
    // for the insertions (2x on the bench's features)
    CU(knn_tc16_pack(h->train64.as<double>(), n, d, false, h->tc_train_rows.p, nullptr, h->tc_flags.as<int>(), c->stream));
    CU(knn_tc16_pack(h->train64.as<double>(), n, d, false, h->tc_train.p, nullptr, h->tc_flags.as<int>(), c->stream,
                     h->prune_perm.as<int>()));
    c->launches++;
    CU(cudaMemcpyAsync(tc_flags, h->tc_flags.p, sizeof tc_flags, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));        // (the plan's host vectors are sources of the copies above)
  }
  int dense_flags[2] = {0, 0};
  if (!h->dp && d <= kKnnDenseMaxDim && std::getenv("DSP_KNN_NO_DENSE") == nullptr) {
    // sequence-feature sizes (compare_feature_methods.py:106-123): split-fp16 operands in tensor-core tile order
    if (h->tpacked.ensure(knn_dense_packed_bytes(n, d, true)) != cudaSuccess ||
        h->tnorm_dense.ensure(sizeof(float) * (size_t)knn_dense_padded_rows(n, true)) != cudaSuccess ||
        h->dense_flags.ensure(64) != cudaSuccess)
      return fail(DSP_ERR_NOMEM, "device allocation failed");
    CU(knn_dense_pack(h->train64.as<double>(), n, d, true, h->tpacked.p, h->tnorm_dense.as<float>(), INFINITY,
                      h->dense_flags.as<int>(), true, c->stream));
    c->launches++;
    CU(cudaMemcpyAsync(dense_flags, h->dense_flags.p, sizeof dense_flags, cudaMemcpyDeviceToHost, c->stream));
  }
  CU(cudaStreamSynchronize(c->stream));
  if (h->tpacked.p) std::memcpy(&h->tnorm_max, &dense_flags[0], sizeof(float));
  if (h->dp) h->scan = h->tc_train.p && tc_flags[1] == 0 ? kScanTc16 : kScanFp32;
  else h->scan = h->tpacked.p && dense_flags[1] == 0 ? kScanDense : kScanF64;
  *out = h.release();
  return DSP_OK;
}

int dsp_knn_fit_host(dsp_context* c, const double* train, const int32_t* labels, int64_t n, int32_t d, int32_t k,
                     int64_t index_base, dsp_knn** out) {
  if (!c || !out || n < 1 || d < 1 || k < 1 || !train || !labels) return fail(DSP_ERR_INVALID, "bad argument");
  if (k > kKnnMaxK) return fail(DSP_ERR_UNSUPPORTED, "n_neighbors > %d is not supported", kKnnMaxK);   // before any copy
  CU(cudaSetDevice(c->device));
  OneShot os(c);
  double* dt = os.dev<double>((size_t)n * d);
  int32_t* dl = os.dev<int32_t>((size_t)n);
  if (!dt || !dl) return fail(DSP_ERR_NOMEM, "device allocation failed");
  CU(cudaMemcpyAsync(dt, train, sizeof(double) * (size_t)n * d, cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(dl, labels, sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice, c->stream));
  return dsp_knn_fit_device(c, dt, dl, n, d, k, index_base, out);
}

int dsp_knn_free(dsp_knn* k) {
  if (!k) return DSP_OK;
  const std::unique_ptr<dsp_knn> owner(k);
  cudaSetDevice(k->ctx->device);
  cudaStreamSynchronize(k->ctx->stream);
  return DSP_OK;
}

int dsp_knn_topk_device(dsp_knn* h, const double* q, int64_t m, int64_t* nbr_idx, double* nbr_sqdist, int32_t* nbr_label) {
  return dsp_knn_topk_bounded_device(h, q, m, nullptr, nbr_idx, nbr_sqdist, nbr_label);
}

// What a candidate stage leaves for the certificate tail of dsp_knn_topk_bounded_device (knn_rerank / knn_refine)
struct KnnStage {
  double err_rel = 0.0, err_floor = 0.0;     // error bound of the candidate scores
  float qnorm_limit = 0.f;                   // > 0: queries with a larger |q|^2 were scored as the zero vector
  const float* thr0 = nullptr;               // per-query start thresholds of the filter
  const double* rerank_bound = nullptr;      // per-query radius the candidates are certified against
  bool allow_short = false;                  // fewer than k rows inside the radius is an answer
  bool redo_all = false;                     // no candidates: every query takes the exhaustive float64 scan
  int refine_cap = 0;                        // rejected queries the second pass (knn_refine) takes
  int launches = 0;
  const unsigned long long* prune_kept = nullptr;    // (DSP_KNN_DEBUG report)
  int64_t prune_visits = 0;
};

// Tensor-core filter.  A query outside its range (|q|^2 above knn_tc16_max_norm(), NaN / inf) is scored as the zero
// vector there and handed to the exhaustive float64 scan by the rerank kernel -- per query, on the device.
static int knn_stage_tc16(dsp_knn* h, const double* q, int64_t m, const double* bound, KnnStage& s) {
  dsp_context* c = h->ctx;
  CU(h->tc_q.ensure(knn_tc16_packed_bytes(m, true)));
  int* qflags = h->tc_flags.as<int>() + 4;
  s.err_rel = knn_dense_err_rel(16);
  s.err_floor = 1.0;
  s.qnorm_limit = knn_tc16_max_norm();
  Tc16Work work;
  const void* tpacked = h->tc_train_rows.p;
  const int unit_q = knn_prune_unit_queries(m, c->sm_count);
  const int64_t visits = (m + unit_q - 1) / unit_q * h->prune_tiles;
  if (c->knn_prune && visits <= INT32_MAX) {          // (the tile lists take units x tiles ints, indexed in int)
    // tile pruning: queries in curve order, a seed pass bounds every query's k-th distance U (capped by the caller's
    // bound), and the main pass visits per unit only the tiles that can hold a row within U; its candidates are
    // certified against U like a bounded call's
    CU(h->prune_ws.ensure(knn_prune_scratch_bytes(m, h->n)));
    CU(h->prune_bound.ensure(sizeof(double) * (size_t)m));
    CU(h->thr0.ensure(sizeof(float) * (size_t)m));
    const unsigned char* pb = h->prune_box.as<unsigned char>();
    const size_t box = sizeof(double) * (size_t)h->prune_tiles * h->d;
    CU(knn_prune_prepare(q, m, h->n, h->d, h->k, h->train64.as<double>(), h->prune_geom.as<KnnPruneGeom>(), h->prune_perm.as<int>(),
                         (const double*)pb, (const double*)(pb + box), (const double*)(pb + 2 * box), h->tc_train.p, h->tc_q.p,
                         h->qnorm.as<float>(), qflags, bound, h->prune_bound.as<double>(), h->cand_idx.as<int>(),
                         h->cand_worst.as<float>(), h->prune_ws.p, c->knn_prune == 1, c->sm_count, c->stream, work));
    tpacked = h->tc_train.p;
    s.rerank_bound = h->prune_bound.as<double>();
    s.prune_kept = work.kept;
    s.prune_visits = visits;
    CU(knn_bound_thresholds(s.rerank_bound, h->qnorm.as<float>(), m, s.err_rel, s.err_floor, h->thr0.as<float>(), c->stream));
    s.thr0 = h->thr0.as<float>();
    s.launches += 12;
  } else {
    CU(knn_tc16_pack(q, m, h->d, true, h->tc_q.p, h->qnorm.as<float>(), qflags, c->stream));
    if (bound) {
      // bounded call (row-sharded KNN): every query's filter starts at the score threshold of its radius
      CU(h->thr0.ensure(sizeof(float) * (size_t)m));
      CU(knn_bound_thresholds(bound, h->qnorm.as<float>(), m, s.err_rel, s.err_floor, h->thr0.as<float>(), c->stream));
      s.thr0 = h->thr0.as<float>();
      s.rerank_bound = bound;
      s.launches += 1;
    }
  }
  CU(knn_tc16_filter(h->tc_q.p, tpacked, m, h->n, h->k, qflags, h->cand_idx.as<int>(), h->cand_worst.as<float>(),
                     c->sm_count, c->stream, s.thr0, work));
  s.launches += 2;
  s.allow_short = bound && s.thr0;
  s.refine_cap = (int)std::min<int64_t>(m, 65536);
  return DSP_OK;
}

int dsp_knn_topk_bounded_device(dsp_knn* h, const double* q, int64_t m, const double* bound, int64_t* nbr_idx, double* nbr_sqdist,
                                int32_t* nbr_label) {
  if (!h || m < 0 || (!q && m)) return fail(DSP_ERR_INVALID, "bad argument");
  if (m == 0) return DSP_OK;
  if (m > INT32_MAX) return fail(DSP_ERR_UNSUPPORTED, "more than 2^31 queries per call");
  dsp_context* c = h->ctx;
  CU(cudaSetDevice(c->device));
  CU(h->redo_list.ensure(sizeof(int32_t) * (size_t)m));
  if (h->scan != kScanF64) {
    CU(h->cand_idx.ensure(sizeof(int) * (size_t)m * kKnnCand));
    CU(h->cand_worst.ensure(sizeof(float) * (size_t)m));
    CU(h->qnorm.ensure(sizeof(float) * (size_t)m));
  }
  // candidates: only the tensor-core filter takes the caller's bound (start thresholds); the other scans ignore it
  KnnStage s;
  if (h->scan == kScanTc16) {
    int rc = knn_stage_tc16(h, q, m, bound, s);
    if (rc) return rc;
  } else if (h->scan == kScanFp32) {
    CU(knn_scan(h->dp, h->train32.as<float>(), h->n, q, m, h->d, h->cand_idx.as<int>(), h->cand_worst.as<float>(),
                h->qnorm.as<float>(), c->stream));
    s.launches = 1;
    s.err_rel = (double)(h->d + 4) * 1.1920929e-7;
    s.refine_cap = (h->dp == 16 && h->k < kKnnCand) ? (int)std::min<int64_t>(m, 65536) : 0;
  } else if (h->scan == kScanDense) {
    // tensor-core candidate scan in chunks of queries (bounded staging); one rerank then certifies all of them
    const int64_t chunk = std::min<int64_t>(m, kKnnDenseQueryChunk);
    CU(h->qpacked.ensure(knn_dense_packed_bytes(chunk, h->d, false)));
    CU(h->qnorm_chunk.ensure(sizeof(float) * (size_t)knn_dense_padded_rows(chunk, false)));
    CU(h->dense_flags.ensure(64));
    for (int64_t q0 = 0; q0 < m; q0 += chunk) {
      const int64_t mc = std::min<int64_t>(chunk, m - q0);
      // the pack kernel writes a norm for every padded row of the chunk: staged, then copied to the queries' slots;
      // the fp16-range flag accumulates over the chunks and is read once (stream order keeps the staging safe)
      CU(knn_dense_pack(q + q0 * h->d, mc, h->d, false, h->qpacked.p, h->qnorm_chunk.as<float>(), 0.f, h->dense_flags.as<int>(),
                        q0 == 0, c->stream));
      CU(cudaMemcpyAsync(h->qnorm.as<float>() + q0, h->qnorm_chunk.p, sizeof(float) * (size_t)mc, cudaMemcpyDeviceToDevice, c->stream));
      CU(knn_dense_scan(h->qpacked.p, h->tpacked.p, h->tnorm_dense.as<float>(), mc, h->n, h->d,
                        h->cand_idx.as<int>() + q0 * kKnnCand, h->cand_worst.as<float>() + q0, c->sm_count, c->stream));
      s.launches += 2;
    }
    int qflags[2] = {0, 0};
    CU(cudaMemcpyAsync(qflags, h->dense_flags.p, sizeof qflags, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    s.redo_all = qflags[1] != 0;     // a query value outside the fp16 range: float64 scan for everything
    s.err_rel = knn_dense_err_rel(h->d);
    s.allow_short = true;
  } else {
    s.redo_all = true;     // feature dimension beyond both scans (or values outside the fp16 range)
  }
  // rejected queries: fp32 threshold scan + float64 ranking of the survivors (knn_refine) for up to refine_cap of them,
  // the exhaustive float64 scan for the rest
  h->refine_cap = s.refine_cap;
  if (s.refine_cap) {
    CU(h->refine_list.ensure(sizeof(int32_t) * (size_t)s.refine_cap));
    CU(h->refine_thr.ensure(sizeof(float) * (size_t)s.refine_cap));
    CU(h->surv_count.ensure(sizeof(int32_t) * (size_t)s.refine_cap));
    CU(h->surv_rows.ensure(sizeof(int32_t) * (size_t)s.refine_cap * knn_refine_survivor_cap()));
  }
  if (s.redo_all) {
    CU(knn_redo_all(h->redo_list.as<int32_t>(), h->redo_count.as<int32_t>(), m, c->stream));
  } else {
    CU(knn_rerank(h->train64.as<double>(), h->train32.as<float>(), h->dp, h->n, q, m, h->d, h->k, h->index_base,
                  h->labels.as<int32_t>(), h->cand_idx.as<int>(), h->cand_worst.as<float>(), h->qnorm.as<float>(),
                  h->tnorm_max, s.err_rel, s.err_floor, nbr_idx, nbr_sqdist, nbr_label, h->redo_list.as<int32_t>(),
                  h->redo_count.as<int32_t>(), c->stream, s.refine_cap ? h->refine_list.as<int32_t>() : nullptr,
                  h->refine_thr.as<float>(), s.refine_cap, s.qnorm_limit, s.rerank_bound, s.thr0, s.allow_short));
  }
  c->launches += s.launches + 1;
  if (s.refine_cap) {
    CU(knn_refine(h->train64.as<double>(), h->train32.as<float>(), h->dp, h->n, q, h->d, h->k, h->index_base,
                  h->labels.as<int32_t>(), h->refine_list.as<int32_t>(), h->refine_thr.as<float>(), s.refine_cap,
                  h->surv_count.as<int32_t>(), h->surv_rows.as<int32_t>(), h->redo_count.as<int32_t>(),
                  h->redo_list.as<int32_t>(), nbr_idx, nbr_sqdist, nbr_label, c->sm_count, c->stream, s.allow_short));
    c->launches += 2;
  }
  CU(h->part_d.ensure(sizeof(double) * (size_t)knn_rescan_grid(c->sm_count) * kKnnMaxK));
  CU(h->part_i.ensure(sizeof(long long) * (size_t)knn_rescan_grid(c->sm_count) * kKnnMaxK));
  CU(knn_rescan(h->train64.as<double>(), h->n, q, h->d, h->k, h->index_base, h->labels.as<int32_t>(),
                h->redo_list.as<int32_t>(), h->redo_count.as<int32_t>(), nbr_idx, nbr_sqdist, nbr_label,
                c->sm_count, h->part_d.as<double>(), h->part_i.as<long long>(), (int)std::min<int64_t>(m, INT32_MAX), c->stream));
  c->launches++;
  if (std::getenv("DSP_KNN_DEBUG")) {
    int32_t cnt[4];
    cudaMemcpyAsync(cnt, h->redo_count.p, sizeof cnt, cudaMemcpyDeviceToHost, c->stream);
    cudaStreamSynchronize(c->stream);
    fprintf(stderr, "[knn] m=%lld n=%lld exhaustive=%d refined=%d refined->exhaustive=%d\n", (long long)m, (long long)h->n, cnt[0],
            std::min(cnt[1], h->refine_cap), cnt[2]);
    if (s.prune_kept) {
      unsigned long long kept = 0;
      cudaMemcpyAsync(&kept, s.prune_kept, sizeof kept, cudaMemcpyDeviceToHost, c->stream);
      cudaStreamSynchronize(c->stream);
      fprintf(stderr, "[knn] prune: tile visits kept=%llu of %lld (%s)\n", kept, (long long)s.prune_visits,
              c->knn_prune == 1 && kept > (unsigned long long)(0.85 * (double)s.prune_visits) ? "every tile walked" : "lists walked");
    }
  }
  return DSP_OK;
}

// ---- MFCC + DTW (self-specified variant, oracle/mfcc_dtw_oracle.py) -------------------------------------
int dsp_mfcc_batch_host(dsp_context* c, const int16_t* samples, const int64_t* offsets, const int32_t* lengths,
                        const int32_t* seg_start, const int32_t* seg_end, int64_t n_utts, const dsp_mfcc_params* p,
                        const float* filterbank, const float* dct, const int64_t* mfcc_offsets, float* mfcc_out,
                        int32_t* n_frames_out) {
  if (!c || !p || n_utts < 0 || (n_utts && (!samples || !offsets || !seg_start || !seg_end || !filterbank || !dct || !mfcc_offsets || !mfcc_out)))
    return fail(DSP_ERR_INVALID, "bad argument");
  int rc = check_mfcc_params(p);
  if (rc) return rc;
  if (n_utts == 0) return DSP_OK;
  CU(cudaSetDevice(c->device));
  int64_t span = 0;
  for (int64_t b = 0; b < n_utts; ++b) span = std::max<int64_t>(span, offsets[b] + (lengths ? lengths[b] : offsets[b + 1] - offsets[b]));
  const int64_t total_frames = mfcc_offsets[n_utts];
  OneShot os(c);
  int16_t* d_s = os.dev<int16_t>((size_t)span);
  int64_t* d_off = os.dev<int64_t>((size_t)n_utts + 1);
  int32_t* d_len = lengths ? os.dev<int32_t>((size_t)n_utts) : nullptr;
  int32_t* d_st = os.dev<int32_t>((size_t)n_utts);
  int32_t* d_en = os.dev<int32_t>((size_t)n_utts);
  int64_t* d_mo = os.dev<int64_t>((size_t)n_utts + 1);
  float* d_out = os.dev<float>((size_t)std::max<int64_t>(total_frames, 1) * p->n_ceps);
  int32_t* d_nf = os.dev<int32_t>((size_t)n_utts);
  if (!d_s || !d_off || (lengths && !d_len) || !d_st || !d_en || !d_mo || !d_out || !d_nf)
    return fail(DSP_ERR_NOMEM, "device allocation failed");
  cudaStream_t st = c->stream;
  CU(cudaMemcpyAsync(d_s, samples, sizeof(int16_t) * (size_t)span, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(d_off, offsets, sizeof(int64_t) * ((size_t)n_utts + 1), cudaMemcpyHostToDevice, st));
  if (lengths) CU(cudaMemcpyAsync(d_len, lengths, sizeof(int32_t) * (size_t)n_utts, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(d_st, seg_start, sizeof(int32_t) * (size_t)n_utts, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(d_en, seg_end, sizeof(int32_t) * (size_t)n_utts, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(d_mo, mfcc_offsets, sizeof(int64_t) * ((size_t)n_utts + 1), cudaMemcpyHostToDevice, st));
  // tables come from the context's cache: a repeated call uploads only its inputs
  rc = dsp_mfcc_batch_device(c, d_s, d_off, d_len, d_st, d_en, n_utts, p, filterbank, dct, d_mo, d_out, d_nf);
  if (rc) return rc;
  if (total_frames > 0) CU(cudaMemcpyAsync(mfcc_out, d_out, sizeof(float) * (size_t)total_frames * p->n_ceps, cudaMemcpyDeviceToHost, st));
  if (n_frames_out) CU(cudaMemcpyAsync(n_frames_out, d_nf, sizeof(int32_t) * (size_t)n_utts, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  return DSP_OK;
}

int dsp_dtw_topk_host(dsp_context* c, const float* q_feats, const int64_t* q_offsets, int64_t nq, const float* t_feats,
                      const int64_t* t_offsets, const int32_t* t_labels, int64_t nt, int32_t dim, int32_t k,
                      int64_t index_base, float* cost_out, double* nbr_cost, int64_t* nbr_idx, int32_t* nbr_label) {
  if (!c || nq < 0 || nt < 1 || dim < 1 || k < 1 || !q_offsets || !t_offsets || (nq && !q_feats) || !t_feats || (nbr_label && !t_labels))
    return fail(DSP_ERR_INVALID, "bad argument");
  if (k > kKnnMaxK) return fail(DSP_ERR_UNSUPPORTED, "k > %d is not supported", kKnnMaxK);
  if (dim > dtw_max_dim()) return fail(DSP_ERR_UNSUPPORTED, "feature dimension > %d is not supported by the DTW kernel", dtw_max_dim());
  if (nq == 0) return DSP_OK;
  int64_t max_q = 0, max_t = 0;
  for (int64_t i = 0; i < nq; ++i) max_q = std::max(max_q, q_offsets[i + 1] - q_offsets[i]);
  for (int64_t i = 0; i < nt; ++i) max_t = std::max(max_t, t_offsets[i + 1] - t_offsets[i]);
  if (max_q > dtw_max_query_frames()) return fail(DSP_ERR_UNSUPPORTED, "query sequences longer than %d frames are not supported", dtw_max_query_frames());
  if (dtw_smem_bytes((int)max_t, dim) > kMaxSmemPerCta) return fail(DSP_ERR_UNSUPPORTED, "template sequence too long for shared memory (%lld frames x %d features)", (long long)max_t, dim);
  CU(cudaSetDevice(c->device));
  OneShot os(c);
  float* d_q = os.dev<float>((size_t)q_offsets[nq] * dim);
  int64_t* d_qo = os.dev<int64_t>((size_t)nq + 1);
  float* d_t = os.dev<float>((size_t)t_offsets[nt] * dim);
  int64_t* d_to = os.dev<int64_t>((size_t)nt + 1);
  int32_t* d_lab = os.dev<int32_t>((size_t)nt);
  float* d_cost = os.dev<float>((size_t)nq * nt);
  double* d_nc = os.dev<double>((size_t)nq * k);
  int64_t* d_ni = os.dev<int64_t>((size_t)nq * k);
  int32_t* d_nl = os.dev<int32_t>((size_t)nq * k);
  if (!d_q || !d_qo || !d_t || !d_to || !d_lab || !d_cost || !d_nc || !d_ni || !d_nl) return fail(DSP_ERR_NOMEM, "device allocation failed");
  cudaStream_t st = c->stream;
  CU(cudaMemcpyAsync(d_q, q_feats, sizeof(float) * (size_t)q_offsets[nq] * dim, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(d_qo, q_offsets, sizeof(int64_t) * ((size_t)nq + 1), cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(d_t, t_feats, sizeof(float) * (size_t)t_offsets[nt] * dim, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(d_to, t_offsets, sizeof(int64_t) * ((size_t)nt + 1), cudaMemcpyHostToDevice, st));
  if (t_labels) CU(cudaMemcpyAsync(d_lab, t_labels, sizeof(int32_t) * (size_t)nt, cudaMemcpyHostToDevice, st));
  else CU(cudaMemsetAsync(d_lab, 0, sizeof(int32_t) * (size_t)nt, st));
  CU(launch_dtw(d_q, d_qo, nq, (int)max_q, d_t, d_to, nt, (int)max_t, dim, d_cost, st));
  CU(launch_dtw_topk(d_cost, nq, nt, k, index_base, d_lab, d_nc, d_ni, d_nl, st));
  c->launches += 2;
  if (cost_out) CU(cudaMemcpyAsync(cost_out, d_cost, sizeof(float) * (size_t)nq * nt, cudaMemcpyDeviceToHost, st));
  if (nbr_cost) CU(cudaMemcpyAsync(nbr_cost, d_nc, sizeof(double) * (size_t)nq * k, cudaMemcpyDeviceToHost, st));
  if (nbr_idx) CU(cudaMemcpyAsync(nbr_idx, d_ni, sizeof(int64_t) * (size_t)nq * k, cudaMemcpyDeviceToHost, st));
  if (nbr_label) CU(cudaMemcpyAsync(nbr_label, d_nl, sizeof(int32_t) * (size_t)nq * k, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  return DSP_OK;
}

int dsp_mfcc_batch_device(dsp_context* c, const int16_t* samples, const int64_t* offsets, const int32_t* lengths,
                          const int32_t* seg_start, const int32_t* seg_end, int64_t n_utts, const dsp_mfcc_params* p,
                          const float* filterbank, const float* dct, const int64_t* mfcc_offsets, float* mfcc_out,
                          int32_t* n_frames_out) {
  if (!c || !p || n_utts < 0 || (n_utts && (!samples || !offsets || !seg_start || !seg_end || !filterbank || !dct || !mfcc_offsets || !mfcc_out)))
    return fail(DSP_ERR_INVALID, "bad argument");
  int rc = check_mfcc_params(p);
  if (rc) return rc;
  if (n_utts == 0) return DSP_OK;
  CU(cudaSetDevice(c->device));
  dsp_context::MfccEntry* t = nullptr;
  rc = ensure_mfcc_tables(c, p, filterbank, dct, &t);
  if (rc) return rc;
  CU(c->mfcc_work.ensure(sizeof(unsigned int)));
  MfccArgs a{p->frame_length, p->frame_shift, p->n_fft, p->n_mels, p->n_ceps, p->pre_emphasis, (float)p->log_floor};
  CU(launch_mfcc(samples, offsets, lengths, seg_start, seg_end, n_utts, a, t->d_win.as<float>(), t->d_tw.as<float2>(),
                 t->d_fb.as<float>(), t->d_range.as<int2>(), t->d_dct.as<float>(), mfcc_offsets, mfcc_out, n_frames_out,
                 c->mfcc_work.as<unsigned int>(), c->sm_count, c->stream));
  c->launches++;
  return DSP_OK;
}

int dsp_dtw_fit_device(dsp_context* c, const float* t_feats, const int64_t* t_offsets, const int32_t* t_lengths,
                       const int32_t* t_labels, int64_t nt, int32_t dim, int32_t k, int64_t index_base, dsp_dtw** out) {
  if (!c || !out || nt < 1 || dim < 1 || k < 1 || !t_offsets) return fail(DSP_ERR_INVALID, "bad argument");
  *out = nullptr;
  if (k > kKnnMaxK) return fail(DSP_ERR_UNSUPPORTED, "k > %d is not supported", kKnnMaxK);
  if (dim > dtw_max_dim()) return fail(DSP_ERR_UNSUPPORTED, "feature dimension > %d is not supported by the DTW kernel", dtw_max_dim());
  if (nt > INT32_MAX) return fail(DSP_ERR_UNSUPPORTED, "more than 2^31 templates per handle");
  CU(cudaSetDevice(c->device));
  // the one synchronisation: template lengths on the host, for the longest template and the extent of the copy
  std::vector<int64_t> off((size_t)nt + 1);
  std::vector<int32_t> len((size_t)nt);
  CU(cudaMemcpyAsync(off.data(), t_offsets, sizeof(int64_t) * off.size(), cudaMemcpyDeviceToHost, c->stream));
  if (t_lengths) CU(cudaMemcpyAsync(len.data(), t_lengths, sizeof(int32_t) * len.size(), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  int64_t extent = 0, max_t = 0;
  for (int64_t i = 0; i < nt; ++i) {
    const int64_t n = t_lengths ? (int64_t)len[(size_t)i] : off[(size_t)i + 1] - off[(size_t)i];
    if (off[(size_t)i] < 0 || n < 0 || n > INT32_MAX) return fail(DSP_ERR_INVALID, "template %lld: bad offset / length", (long long)i);
    len[(size_t)i] = (int32_t)n;
    max_t = std::max(max_t, n);
    extent = std::max(extent, off[(size_t)i] + n);
  }
  if (extent > 0 && !t_feats) return fail(DSP_ERR_INVALID, "bad argument");
  const size_t per_warp = dtw_fused_smem_per_warp((int)max_t, dim);
  if (per_warp > c->smem_optin)
    return fail(DSP_ERR_UNSUPPORTED, "template sequence too long for shared memory (%lld frames x %d features)", (long long)max_t, dim);
  auto h = std::make_unique<dsp_dtw>();
  h->ctx = c; h->nt = nt; h->index_base = index_base; h->dim = dim; h->k = k; h->max_t = (int)max_t;
  h->warps = (int)std::min<size_t>(dtw_fused_max_warps(), c->smem_optin / per_warp);
  h->h_len = std::move(len);
  if (h->feats.ensure(sizeof(float) * (size_t)std::max<int64_t>(extent, 1) * dim) != cudaSuccess ||
      h->offsets.ensure(sizeof(int64_t) * (size_t)nt) != cudaSuccess || h->t_len.ensure(sizeof(int32_t) * (size_t)nt) != cudaSuccess ||
      h->labels.ensure(sizeof(int32_t) * (size_t)nt) != cudaSuccess || h->stats.ensure(2 * sizeof(unsigned long long)) != cudaSuccess)
    return fail(DSP_ERR_NOMEM, "device allocation failed");
  if (extent > 0) CU(cudaMemcpyAsync(h->feats.p, t_feats, sizeof(float) * (size_t)extent * dim, cudaMemcpyDeviceToDevice, c->stream));
  CU(cudaMemcpyAsync(h->offsets.p, t_offsets, sizeof(int64_t) * (size_t)nt, cudaMemcpyDeviceToDevice, c->stream));
  CU(cudaMemcpyAsync(h->t_len.p, h->h_len.data(), sizeof(int32_t) * (size_t)nt, cudaMemcpyHostToDevice, c->stream));
  if (t_labels) CU(cudaMemcpyAsync(h->labels.p, t_labels, sizeof(int32_t) * (size_t)nt, cudaMemcpyDeviceToDevice, c->stream));
  else CU(cudaMemsetAsync(h->labels.p, 0, sizeof(int32_t) * (size_t)nt, c->stream));
  CU(cudaMemsetAsync(h->stats.p, 0, 2 * sizeof(unsigned long long), c->stream));
  *out = h.release();
  return DSP_OK;
}

int dsp_dtw_topk_device(dsp_dtw* h, const float* q_feats, const int64_t* q_offsets, const int32_t* q_lengths, int64_t nq,
                        int32_t max_q_frames, double* nbr_cost, int64_t* nbr_idx, int32_t* nbr_label) {
  return dsp_dtw_topk_bounded_device(h, q_feats, q_offsets, q_lengths, nq, max_q_frames, nullptr, nbr_cost, nbr_idx, nbr_label);
}

int dsp_dtw_topk_bounded_device(dsp_dtw* h, const float* q_feats, const int64_t* q_offsets, const int32_t* q_lengths, int64_t nq,
                                int32_t max_q_frames, const double* bound_cost, double* nbr_cost, int64_t* nbr_idx,
                                int32_t* nbr_label) {
  if (!h || nq < 0 || (nq && !q_offsets)) return fail(DSP_ERR_INVALID, "bad argument");   // q_feats: NULL when every query is empty
  dsp_context* c = h->ctx;
  CU(cudaSetDevice(c->device));
  const int slices = dtw_fused_slices(nq, h->nt, c->sm_count);
  const size_t cand = (size_t)dtw_fused_units(nq, c->sm_count) * h->k;   // >= nq * slices * k
  if (nq > 0) {
    CU(h->cand_d.ensure(sizeof(float) * cand));
    CU(h->cand_i.ensure(sizeof(int64_t) * cand));
  }
  CU(launch_dtw_topk_fused(q_feats, q_offsets, q_lengths, nq, max_q_frames, h->feats.as<float>(), h->offsets.as<int64_t>(),
                           h->t_len.as<int32_t>(), h->nt, h->max_t, h->dim, h->k, bound_cost, slices, h->warps, h->index_base,
                           h->labels.as<int32_t>(), h->cand_d.as<float>(), h->cand_i.as<int64_t>(),
                           h->stats.as<unsigned long long>(), nbr_cost, nbr_idx, nbr_label, c->stream));
  c->launches += nq > 0 ? 3 : 1;
  return DSP_OK;
}

int dsp_dtw_last_stats(dsp_dtw* h, int64_t* pairs_scored, int64_t* pairs_abandoned) {
  if (!h) return fail(DSP_ERR_INVALID, "bad argument");
  CU(cudaSetDevice(h->ctx->device));
  unsigned long long cnt[2] = {0, 0};
  CU(cudaMemcpyAsync(cnt, h->stats.p, sizeof cnt, cudaMemcpyDeviceToHost, h->ctx->stream));
  CU(cudaStreamSynchronize(h->ctx->stream));
  if (pairs_scored) *pairs_scored = (int64_t)cnt[0];
  if (pairs_abandoned) *pairs_abandoned = (int64_t)cnt[1];
  return DSP_OK;
}

int dsp_dtw_free(dsp_dtw* h) {
  if (!h) return DSP_OK;
  const std::unique_ptr<dsp_dtw> owner(h);
  cudaSetDevice(h->ctx->device);
  cudaStreamSynchronize(h->ctx->stream);
  return DSP_OK;
}

int dsp_knn_last_stats(dsp_knn* h, int64_t* rescanned, int32_t* scan_kind) {
  if (!h) return fail(DSP_ERR_INVALID, "bad argument");
  CU(cudaSetDevice(h->ctx->device));
  // queries the first certificate rejected: refined ([1], up to the list's capacity: a query past it took a slot number
  // there, then went to the exhaustive scan) + sent straight to the exhaustive scan ([0] minus those the refinement
  // passed on, [2])
  int32_t cnt[4] = {0, 0, 0, 0};
  if (h->redo_count.p) {
    CU(cudaMemcpyAsync(cnt, h->redo_count.p, sizeof cnt, cudaMemcpyDeviceToHost, h->ctx->stream));
    CU(cudaStreamSynchronize(h->ctx->stream));
  }
  if (rescanned) *rescanned = (int64_t)cnt[0] + std::min(cnt[1], h->refine_cap) - cnt[2];
  if (scan_kind) *scan_kind = h->scan;
  return DSP_OK;
}

int dsp_knn_predict_device(dsp_knn* h, const double* q, int64_t m, int32_t* labels_out) {
  if (!h || !labels_out) return fail(DSP_ERR_INVALID, "bad argument");
  if (m == 0) return DSP_OK;
  dsp_context* c = h->ctx;
  CU(cudaSetDevice(c->device));
  CU(h->nbr_label.ensure(sizeof(int32_t) * (size_t)m * h->k));
  int rc = dsp_knn_topk_device(h, q, m, nullptr, nullptr, h->nbr_label.as<int32_t>());
  if (rc) return rc;
  CU(knn_vote(h->nbr_label.as<int32_t>(), m, h->k, labels_out, c->stream));
  c->launches++;
  return DSP_OK;
}

int dsp_knn_topk_host(dsp_knn* h, const double* q, int64_t m, int64_t* nbr_idx, double* nbr_sqdist, int32_t* nbr_label) {
  if (!h || m < 0 || (!q && m)) return fail(DSP_ERR_INVALID, "bad argument");
  if (m == 0) return DSP_OK;
  dsp_context* c = h->ctx;
  CU(cudaSetDevice(c->device));
  CU(h->q.ensure(sizeof(double) * (size_t)m * h->d));
  CU(h->o_idx.ensure(sizeof(int64_t) * (size_t)m * h->k));
  CU(h->o_dist.ensure(sizeof(double) * (size_t)m * h->k));
  CU(h->o_lab.ensure(sizeof(int32_t) * (size_t)m * h->k));
  CU(cudaMemcpyAsync(h->q.p, q, sizeof(double) * (size_t)m * h->d, cudaMemcpyHostToDevice, c->stream));
  int rc = dsp_knn_topk_device(h, h->q.as<double>(), m, h->o_idx.as<int64_t>(), h->o_dist.as<double>(), h->o_lab.as<int32_t>());
  if (rc) return rc;
  if (nbr_idx) CU(cudaMemcpyAsync(nbr_idx, h->o_idx.p, sizeof(int64_t) * (size_t)m * h->k, cudaMemcpyDeviceToHost, c->stream));
  if (nbr_sqdist) CU(cudaMemcpyAsync(nbr_sqdist, h->o_dist.p, sizeof(double) * (size_t)m * h->k, cudaMemcpyDeviceToHost, c->stream));
  if (nbr_label) CU(cudaMemcpyAsync(nbr_label, h->o_lab.p, sizeof(int32_t) * (size_t)m * h->k, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return DSP_OK;
}

int dsp_knn_predict_host(dsp_knn* h, const double* q, int64_t m, int32_t* labels_out) {
  if (!h || !labels_out || m < 0 || (!q && m)) return fail(DSP_ERR_INVALID, "bad argument");
  if (m == 0) return DSP_OK;
  dsp_context* c = h->ctx;
  CU(cudaSetDevice(c->device));
  CU(h->q.ensure(sizeof(double) * (size_t)m * h->d));
  CU(h->o_lab.ensure(sizeof(int32_t) * (size_t)m));
  CU(cudaMemcpyAsync(h->q.p, q, sizeof(double) * (size_t)m * h->d, cudaMemcpyHostToDevice, c->stream));
  int rc = dsp_knn_predict_device(h, h->q.as<double>(), m, h->o_lab.as<int32_t>());
  if (rc) return rc;
  CU(cudaMemcpyAsync(labels_out, h->o_lab.p, sizeof(int32_t) * (size_t)m, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return DSP_OK;
}

int dsp_knn_merge_vote_device(dsp_context* c, const double* cand_sqdist, const int64_t* cand_idx, const int32_t* cand_label,
                              int32_t n_lists, int64_t m, int32_t k, int32_t* labels_out, int64_t* nbr_idx_out,
                              double* nbr_sqdist_out) {
  if (!c || !cand_sqdist || !cand_idx || !cand_label || n_lists < 1 || m < 0 || k < 1 || k > kKnnMaxK)
    return fail(DSP_ERR_INVALID, "bad argument");
  CU(cudaSetDevice(c->device));
  CU(knn_merge_vote(cand_sqdist, cand_idx, cand_label, n_lists, m, k, labels_out, nbr_idx_out, nbr_sqdist_out, c->stream));
  c->launches++;
  return DSP_OK;
}

}  // extern "C"
