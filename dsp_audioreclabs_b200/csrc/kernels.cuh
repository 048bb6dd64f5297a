// Kernel argument blocks and launch-visible declarations (internal to libdspfront).
#pragma once
#include "common.cuh"

namespace dsp {

constexpr int kExactThreads = 256;

// Feature framing rule of frame_signal (audio_processing.py:320-331) in closed form:
// frames start at k*fs while k*fs < n, stopping after the first frame that reaches n.
__host__ __device__ inline int64_t frame_count_host_device(int64_t n, int64_t fl, int64_t fs) {
  if (n <= 0) return 0;
  const int64_t a = (n + fs - 1) / fs;
  const int64_t rem = n > fl ? n - fl : 0;
  const int64_t b = (rem + fs - 1) / fs + 1;
  return a < b ? a : b;
}

struct ExactArgs {
  const void* samples;
  int dtype, channels;
  const int64_t* offsets;       // [B+1] element offsets
  const int32_t* lengths;       // [B] elements per utterance, or null = offsets[b+1] - offsets[b]
  const int64_t* feat_offsets;  // [B+1] or null (single utterance: 0)
  const int64_t* epd_offsets;   // [B+1] or null
  const int32_t* list;          // utterance indices to process, or null = 0..n_items-1
  const int32_t* list_count;    // device count of `list`, or null = n_items
  int64_t n_items;
  int fl, fs;
  int do_epd, pre_mode /* bit0 remove_dc, bit1 normalize */, do_features;
  double hr, lr, zr;
  const double* win;            // [fl] float64 window
  double* zbuf;                 // per-CTA scratch for the pre-processed signal
  int64_t zbuf_stride;
  double* seqbuf;               // per-CTA scratch: 5 arrays of seq_cap doubles
  int64_t seq_cap;
  dsp_frontend_outputs out;
  double* pre_out;              // optional: pre-processed signal (single-utterance calls)
  double* frames_out;           // optional: dense [F, fl] windowed frames
  double* epd_zcr_f64;          // optional float64 zcr_list
  double* feat_f64[3];          // optional float64 energy / magnitude / zcr
  double* stats_f64;            // optional float64 [B,15]
};

struct PcmArgs {
  const int16_t* samples;
  const int64_t* offsets;
  const int32_t* lengths;       // [B] or null (packed CSR)
  const int64_t* feat_offsets;
  const int64_t* epd_offsets;
  int64_t n_utts;
  int fl, fs, window, do_epd;
  double hr, lr, zr;
  const float* win_f32;         // [fl] window as float
  int cap_samples;              // shared-memory capacity in samples (multiple of 64)
  int cap_frames;               // capacity for per-frame arrays
  int tma_chunk;                // bytes per bulk copy (multiple of 16)
  int stagger_ns;               // start-up delay per co-resident CTA index (0 = none)
  int sm_count;
  int ring_slots, n_rec, cap_groups;   // frontend_pipe_kernel: shared-memory plan (pipe_kernel_plan)
  long long* prof;              // debug: per-phase cycle counters (NULL normally)
  unsigned int* work_counter;   // dynamic utterance scheduler
  int32_t* flag_list;           // utterances that need the float64 replay
  int32_t* flag_count;
  dsp_frontend_outputs out;
};

__global__ void frontend_exact_kernel(const ExactArgs a);
__global__ void frame_features_kernel(const double* frames, int64_t n_frames, int fl, double* energy,
                                      double* magnitude, double* zcr);
__global__ void sequence_stats_kernel(const double* s0, const double* s1, const double* s2, int n,
                                      double* out);

// frontend_pcm.cu
size_t pcm_kernel_smem_bytes(int cap_samples, int cap_frames, int fl, bool resident);
cudaError_t launch_frontend_pcm(int variant, const PcmArgs& a, int grid, size_t smem, cudaStream_t st);
int pcm_kernel_max_ctas_per_sm(int variant, size_t smem, size_t smem_optin);   // 0: the build does not fit
int pcm_num_variants();
// frontend_pipe.cu
struct PipePlan { int ring_slots, n_rec, cap_groups; size_t smem; };
bool pipe_kernel_plan(int64_t max_len, int cap_frames, int fl, size_t smem_limit, PipePlan* plan);
cudaError_t launch_frontend_pipe(const PcmArgs& a, int grid, size_t smem, cudaStream_t st);
bool pcm_variant_streams(int variant);

}  // namespace dsp
