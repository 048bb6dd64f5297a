// MFCC + DTW launchers (internal to libdspfront; csrc/mfcc_dtw.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace dsp {

struct MfccArgs {
  int frame_length, frame_shift, n_fft, n_mels, n_ceps;
  double pre_emphasis;
  float log_floor;
};

size_t mfcc_smem_bytes(int n_fft, int n_mels);
cudaError_t launch_mfcc(const int16_t* samples, const int64_t* offsets, const int32_t* lengths, const int32_t* seg_start,
                        const int32_t* seg_end, int64_t n_utts, const MfccArgs& a, const float* window, const float2* twiddle,
                        const float* filterbank, const int2* fb_range, const float* dct, const int64_t* mfcc_offsets, float* out,
                        int32_t* n_frames_out, unsigned int* work_counter, int sm_count, cudaStream_t st);
int dtw_max_query_frames();
int dtw_max_dim();
size_t dtw_smem_bytes(int max_t_frames, int dim);     // template frames + one boundary row
cudaError_t launch_dtw(const float* qf, const int64_t* qoff, int64_t nq, int max_q_frames, const float* tf, const int64_t* toff,
                       int64_t nt, int max_t_frames, int dim, float* cost, cudaStream_t st);
// fused DTW + top k over resident templates (no cost matrix): qlen / tlen give sequence lengths (qlen may be NULL:
// offsets[i + 1] - offsets[i]); max_q_frames only picks the strip height (<= 0: unknown); bound (nullable, float64
// [nq]) keeps only templates with cost <= bound, none where it is not >= 0.  cand_d / cand_i hold
// nq * slices * k entries, stats two counters (pairs scored, pairs abandoned).  Warps per CTA: up to
// dtw_fused_max_warps(), each with dtw_fused_smem_per_warp() bytes of shared memory.
size_t dtw_fused_smem_per_warp(int max_t_frames, int dim);
int dtw_fused_max_warps();
int64_t dtw_fused_units(int64_t nq, int sm_count);                  // upper bound of nq * dtw_fused_slices(nq, ...)
int dtw_fused_slices(int64_t nq, int64_t nt, int sm_count);
cudaError_t launch_dtw_topk_fused(const float* qf, const int64_t* qoff, const int32_t* qlen, int64_t nq, int max_q_frames,
                                  const float* tf, const int64_t* toff, const int32_t* tlen, int64_t nt, int max_t_frames, int dim,
                                  int k, const double* bound, int slices, int warps, int64_t index_base, const int32_t* labels,
                                  float* cand_d, int64_t* cand_i, unsigned long long* stats, double* nbr_cost,
                                  int64_t* nbr_idx, int32_t* nbr_label, cudaStream_t st);
cudaError_t launch_dtw_topk(const float* cost, int64_t nq, int64_t nt, int k, int64_t index_base, const int32_t* labels,
                            double* nbr_cost, int64_t* nbr_idx, int32_t* nbr_label, cudaStream_t st);

}  // namespace dsp
