// KNN launchers (internal to libdspfront).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <vector>

namespace dsp {

constexpr int kKnnCand = 8;    // fp32 candidates kept per query by the scan
constexpr int kKnnMaxK = 16;   // largest supported n_neighbors (certificate needs k < kKnnCand, else rescan)

int knn_padded_dim(int d);     // 16 / 32 / 64, or 0 when d is too large for the tiled scan
cudaError_t knn_pack(const double* train, int64_t n, int d, int dp, float* train32, float* tnorm_max,
                     cudaStream_t st);
cudaError_t knn_scan(int dp, const float* train32, int64_t n, const double* q, int64_t m, int d,
                     int* cand_idx, float* cand_worst, float* qnorm, cudaStream_t st);
cudaError_t knn_rerank(const double* train, const float* train32, int dp, int64_t n, const double* q,
                       int64_t m, int d, int k, int64_t index_base, const int32_t* labels,
                       const int* cand_idx, const float* cand_worst, const float* qnorm,
                       float tnorm_max_host, double err_rel, double err_floor, int64_t* nbr_idx, double* nbr_sqdist, int32_t* nbr_label,
                       int32_t* redo_list, int32_t* redo_count, cudaStream_t st, int32_t* refine_list = nullptr,
                       float* refine_thr = nullptr, int refine_cap = 0, float qnorm_limit = 0.f,
                       const double* bound = nullptr, const float* thr0 = nullptr, bool allow_short = true);
// D <= 15: second pass for the queries the certificate rejected (fp32 threshold scan + float64 ranking of the survivors);
// counts = redo_count: [0] exhaustive rescans, [1] refined queries, [2] refined queries passed on to the exhaustive scan
int knn_refine_survivor_cap();
cudaError_t knn_refine(const double* train, const float* train32, int dp, int64_t n, const double* q, int d, int k,
                       int64_t index_base, const int32_t* labels, const int32_t* refine_list, const float* refine_thr,
                       int refine_cap, int32_t* surv_count, int32_t* surv_rows, int32_t* counts, int32_t* redo_list,
                       int64_t* nbr_idx, double* nbr_sqdist, int32_t* nbr_label, int sm_count, cudaStream_t st,
                       bool allow_short = false);
cudaError_t knn_redo_all(int32_t* redo_list, int32_t* redo_count, int64_t m, cudaStream_t st);
cudaError_t knn_rescan(const double* train, int64_t n, const double* q, int d, int k, int64_t index_base,
                       const int32_t* labels, const int32_t* redo_list, const int32_t* redo_count,
                       int64_t* nbr_idx, double* nbr_sqdist, int32_t* nbr_label, int sm_count,
                       double* part_d, long long* part_i, int max_redo, cudaStream_t st);
// wide features (d > 64): the rows of a rejected query are split over several CTAs when few queries were rejected;
// part_d / part_i hold knn_rescan_grid(sm_count) * kKnnMaxK partial results each
int knn_rescan_grid(int sm_count);
cudaError_t knn_vote(const int32_t* nbr_label, int64_t m, int k, int32_t* out, cudaStream_t st);
cudaError_t knn_merge_vote(const double* cd, const int64_t* ci, const int32_t* cl, int r, int64_t m,
                           int k, int32_t* labels_out, int64_t* idx_out, double* dist_out,
                           cudaStream_t st);

// knn_tc16.cu: tensor-core candidate filter for d <= 15 (one K = 16 MMA step, |t|^2 as the 16th feature)
float knn_tc16_max_norm();                                   // largest |x|^2 the filter accepts (else: fp32 scan)
int64_t knn_tc16_padded_rows(int64_t rows, bool query);
size_t knn_tc16_packed_bytes(int64_t rows, bool query);
constexpr int kTc16TileRows = 128;                           // train rows per filter tile
constexpr int kTc16UnitQueries = 256;                        // queries per filter work unit
// flags[0] = max |x|^2 (float bits), flags[1] = 1 when a row is outside the range; norms (optional): |x|^2 per row,
// at the source row; gather (optional): packed row r holds source row gather[r]
cudaError_t knn_tc16_pack(const double* x, int64_t rows, int d, bool query, void* packed, float* norms, int* flags, cudaStream_t st,
                          const int* gather = nullptr);
// What the filter walks and how its positions map back.  Default: every work unit in turn, every train tile in order,
// packed positions = row / query indices.
struct Tc16Work {
  const int* tiles = nullptr;        // [units][stride]: the train tiles each unit visits (nullptr: all of them)
  const int* tile_count = nullptr;   // [units]
  int stride = 0;
  const int* unit_order = nullptr;   // units in the order they are claimed (nullptr: 0, 1, ...)
  int* counter = nullptr;            // claim counter, zero at launch (nullptr: static stride over the grid)
  const unsigned long long* kept = nullptr;   // (optional, device) tile visits of all lists: above kept_limit, walk every tile
  unsigned long long kept_limit = 0;
  const int* qperm = nullptr;        // packed query position -> query index
  const int* tperm = nullptr;        // packed train position -> train row
};
// k: neighbours the caller will certify (the filter keeps k + 2 candidates for k <= 3, else 8); needs n >= 64
// thr0 (optional, [m], by query index): start every query's filter at this score threshold (knn_bound_thresholds)
cudaError_t knn_tc16_filter(const void* qpacked, const void* tpacked, int64_t m, int64_t n, int k, const int* qflags, int* cand_idx,
                            float* cand_worst, int sm_count, cudaStream_t st, const float* thr0 = nullptr, const Tc16Work& work = Tc16Work());

// Tile pruning for the filter (knn_tc16.cu).  At fit the train rows are ordered into 128-row tiles by recursive median
// splits along their principal axes, and every tile keeps its bounding box in those axes.  Per call the queries are
// sorted along a space-filling curve into 256-query units; a seed pass over each unit's nearest tiles bounds every
// query's k-th distance U, and a unit visits only the tiles whose box lies within max U of its own box.
constexpr int kPruneMaxDim = 15;
constexpr int kPruneSeedTiles = 4;                           // tiles per unit in the seed pass
struct KnnPruneGeom {
  int d;
  double mean[kPruneMaxDim];
  double axis[kPruneMaxDim][kPruneMaxDim];                   // principal axes, largest variance first: axis[a][j]
  double key_lo[3], key_scale[3];                            // curve quantisation of the first three projections
};
struct KnnPrunePlan {
  KnnPruneGeom geom;
  std::vector<int> perm;                                     // tile-ordered position -> train row
  std::vector<double> lo, hi, slack;                         // per tile: [tiles][d] box in the axes, rounding slack
};
void knn_prune_plan(const double* train, int64_t n, int d, KnnPrunePlan& plan);      // host, float64
// device scratch of one call: knn_prune_scratch_bytes() bytes, 256-byte aligned
size_t knn_prune_scratch_bytes(int64_t m, int64_t n);
// Builds the query order, packs the queries, runs the seed pass and leaves the main pass's tile lists: bound[m] = U per
// query (min with caller_bound when given), work = the schedule of the main filter call.  auto_fallback: the main pass
// walks every tile when the lists keep more than 85 % of all tile visits.
cudaError_t knn_prune_prepare(const double* q, int64_t m, int64_t n, int d, int k, const double* train, const KnnPruneGeom* geom,
                              const int* tperm, const double* tile_lo, const double* tile_hi, const double* tile_slack, const void* tpacked,
                              void* qpacked, float* qnorm, int* qflags, const double* caller_bound, double* bound, int* cand_idx,
                              float* cand_worst, void* scratch, bool auto_fallback, int sm_count, cudaStream_t st, Tc16Work& work);
// bound[i] = an upper bound on query i's k-th squared distance (exact arithmetic) -> thr0[i] = the score threshold below
// which every row that can still matter is guaranteed to fall (bound - |q|^2 + twice the scan's error at that radius)
cudaError_t knn_bound_thresholds(const double* bound, const float* qnorm, int64_t m, double err_rel, double err_floor, float* thr0,
                                 cudaStream_t st);

// knn_dense.cu: tensor-core candidate scan for feature dimensions beyond the tiled scan (sequence features, D = 2 * max_len)
int knn_dense_kblocks(int d);
int64_t knn_dense_padded_rows(int64_t rows, bool train);      // rows rounded up to the tile height (queries 128, train 256)
size_t knn_dense_packed_bytes(int64_t rows, int d, bool train);
// norms: one float per PADDED row.  flags[0] = max |x|^2 as float bits, flags[1] = 1 when a value does not fit fp16
// (the caller falls back to the float64 scan); reset_flags = false accumulates over several calls
cudaError_t knn_dense_pack(const double* x, int64_t rows, int d, bool train, void* packed, float* norms, float pad_norm,
                           int* flags, bool reset_flags, cudaStream_t st);
cudaError_t knn_dense_scan(const void* qpacked, const void* tpacked, const float* tnorm, int64_t m, int64_t n, int d,
                           int* cand_idx, float* cand_worst, int sm_count, cudaStream_t st);
// bound on |score_scan - score_exact| / (|q| + |t|max)^2 for the split-fp16 tensor-core evaluation: 3 * D / 16 fp32
// accumulations of K = 16 partial sums, the dropped lo*lo term, the fp32 norms and the final multiply-add
inline double knn_dense_err_rel(int d) { return (3.0 * d / 16.0 + 32.0) * 2.384185791015625e-07; }

}  // namespace dsp
