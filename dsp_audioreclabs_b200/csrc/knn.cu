// KNN classify (src/models.py:33-35,52-58 -> sklearn KNeighborsClassifier(n_neighbors=k),
// Euclidean, uniform vote; SURVEY.md section 3.3).
//
// The reference's result is the k train rows with the smallest float64 distance and a
// majority vote with ties to the smallest label.  The feature dimension of this path is
// 15 (pad 16): far too thin for a tensor-core contraction to be "genuinely dense", so the
// scan is a shared-memory tiled fp32 kernel:
//
//   scan    each thread keeps QPT queries in registers (pre-scaled by -2) and streams train
//           tiles staged in shared memory ([t_0..t_{D-1}, |t|^2] per row, broadcast loads);
//           per pair it is D FMAs starting from |t|^2, then one compare against the worst of
//           a sorted register list of KC candidates.  The train matrix is never re-read from
//           HBM per query and the m x n distance matrix is never materialised.
//   rerank  float64 direct-form distances sum_j (q_j - t_j)^2 (the kd-tree's accumulation
//           order) for the KC candidates, sorted by (distance, index); the top k are CERTIFIED
//           exact when the k-th exact distance is below the worst kept fp32 score minus a
//           bound on the fp32 error -- otherwise the query is rescanned exhaustively in
//           float64 (rescan kernel), so labels never depend on fp32 rounding.
#include <algorithm>
#include "kernels.cuh"
#include "knn.cuh"

namespace dsp {

namespace {

constexpr int kScanThreads = 128;
constexpr int kTileRows = 128;

template <int KC>
__device__ __forceinline__ void cand_insert(float (&cd)[KC], int (&ci)[KC], float d, int idx) {
  // sorted ascending; cd[KC-1] is the worst kept score
  if (d < cd[KC - 1]) {
    cd[KC - 1] = d; ci[KC - 1] = idx;
#pragma unroll
    for (int s = KC - 1; s > 0; --s) {
      if (cd[s] < cd[s - 1]) {
        const float td = cd[s]; cd[s] = cd[s - 1]; cd[s - 1] = td;
        const int ti = ci[s]; ci[s] = ci[s - 1]; ci[s - 1] = ti;
      }
    }
  }
}

// fp32 candidate scan.  train32: [n, DP] rows of (t_0..t_{D-1}, 0.., |t|^2 at DP-1) -- |t|^2 rounded
// to float.  queries: float64 [m, d].  Outputs KC candidate indices per query and the worst
// kept score.
template <int DP, int QPT>
__global__ void __launch_bounds__(kScanThreads)
knn_scan_kernel(const float* __restrict__ train32, int64_t n, const double* __restrict__ queries,
                int64_t m, int d, int* __restrict__ cand_idx, float* __restrict__ cand_worst,
                float* __restrict__ qnorm_out) {
  __shared__ __align__(16) float tile[kTileRows * DP];
  const int64_t q0 = ((int64_t)blockIdx.x * kScanThreads + threadIdx.x) * QPT;
  float q[QPT][DP - 1];
  float cd[QPT][kKnnCand];
  int ci[QPT][kKnnCand];
#pragma unroll
  for (int r = 0; r < QPT; ++r) {
    float nn = 0.f;
#pragma unroll
    for (int j = 0; j < DP - 1; ++j) {
      const float v = (q0 + r < m && j < d) ? (float)queries[(q0 + r) * d + j] : 0.f;
      nn = fmaf(v, v, nn);
      q[r][j] = -2.f * v;
    }
    if (q0 + r < m) qnorm_out[q0 + r] = nn;
#pragma unroll
    for (int c = 0; c < kKnnCand; ++c) { cd[r][c] = INFINITY; ci[r][c] = -1; }
  }
  for (int64_t base = 0; base < n; base += kTileRows) {
    const int rows = (int)min((int64_t)kTileRows, n - base);
    __syncthreads();
    {
      const float4* src = reinterpret_cast<const float4*>(train32 + base * DP);
      float4* dst = reinterpret_cast<float4*>(tile);
      for (int i = threadIdx.x; i < rows * (DP / 4); i += kScanThreads) dst[i] = src[i];
    }
    __syncthreads();
    for (int j = 0; j < rows; ++j) {
      const float4* row = reinterpret_cast<const float4*>(tile + j * DP);
      float acc[QPT];
      const float tn = tile[j * DP + DP - 1];
#pragma unroll
      for (int r = 0; r < QPT; ++r) acc[r] = tn;
#pragma unroll
      for (int v = 0; v < DP / 4; ++v) {
        const float4 x = row[v];
#pragma unroll
        for (int r = 0; r < QPT; ++r) {
          acc[r] = fmaf(q[r][4 * v], x.x, acc[r]);
          acc[r] = fmaf(q[r][4 * v + 1], x.y, acc[r]);
          acc[r] = fmaf(q[r][4 * v + 2], x.z, acc[r]);
          if (4 * v + 3 < DP - 1) acc[r] = fmaf(q[r][4 * v + 3], x.w, acc[r]);
        }
      }
#pragma unroll
      for (int r = 0; r < QPT; ++r) cand_insert<kKnnCand>(cd[r], ci[r], acc[r], (int)(base + j));
    }
  }
#pragma unroll
  for (int r = 0; r < QPT; ++r) {
    if (q0 + r < m) {
#pragma unroll
      for (int c = 0; c < kKnnCand; ++c) cand_idx[(q0 + r) * kKnnCand + c] = ci[r][c];
      cand_worst[q0 + r] = cd[r][kKnnCand - 1];
    }
  }
}

// The D <= 15 scan on packed fp32x2 arithmetic (sm_100 FFMA2): a thread scores TWO train rows per instruction.  The
// tile is staged as row pairs interleaved column by column, so one broadcast LDS.128 delivers two (row j, row j + 1)
// operand pairs as aligned 64-bit register pairs; the query coefficients sit in registers as (q, q) pairs.  FFMA2 has
// the FMA throughput of FFMA at half the issue slots: the scalar kernel needs 41 issue slots for the 30 FMAs of a
// (row, 2 queries) step, this one 46 for 60.  Same operations in the same order: bit-identical scores.
typedef unsigned long long f32x2_t;
__device__ __forceinline__ f32x2_t pk2f(float a, float b) { f32x2_t r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ void unpk2f(f32x2_t v, float& a, float& b) { asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); }
__device__ __forceinline__ f32x2_t fma2f(f32x2_t a, f32x2_t b, f32x2_t c) { f32x2_t d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }

constexpr int kPairQpt = 2;
__global__ void __launch_bounds__(kScanThreads)
knn_scan_pair_kernel(const float* __restrict__ train32, int64_t n, const double* __restrict__ queries,
                     int64_t m, int d, int* __restrict__ cand_idx, float* __restrict__ cand_worst,
                     float* __restrict__ qnorm_out) {
  constexpr int DP = 16;
  __shared__ __align__(16) float tile[kTileRows * DP];            // [row pair][column][2]
  const int64_t q0 = ((int64_t)blockIdx.x * kScanThreads + threadIdx.x) * kPairQpt;
  f32x2_t qq[kPairQpt][DP - 1];
  float cd[kPairQpt][kKnnCand];
  int ci[kPairQpt][kKnnCand];
#pragma unroll
  for (int r = 0; r < kPairQpt; ++r) {
    float nn = 0.f;
#pragma unroll
    for (int j = 0; j < DP - 1; ++j) {
      const float v = (q0 + r < m && j < d) ? (float)queries[(q0 + r) * d + j] : 0.f;
      nn = fmaf(v, v, nn);
      qq[r][j] = pk2f(-2.f * v, -2.f * v);
    }
    if (q0 + r < m) qnorm_out[q0 + r] = nn;
#pragma unroll
    for (int c = 0; c < kKnnCand; ++c) { cd[r][c] = INFINITY; ci[r][c] = -1; }
  }
  for (int64_t base = 0; base < n; base += kTileRows) {
    const int rows = (int)min((int64_t)kTileRows, n - base);
    const int pairs = (rows + 1) >> 1;
    __syncthreads();
    {
      const float4* src = reinterpret_cast<const float4*>(train32 + base * DP);
      for (int i = threadIdx.x; i < 2 * pairs * (DP / 4); i += kScanThreads) {
        const int row = i >> 2, c4 = (i & 3) * 4;
        // a missing second row of the last pair scores +inf (norm column) and is never kept
        const float4 v = row < rows ? src[i] : make_float4(0.f, 0.f, 0.f, c4 == 12 ? INFINITY : 0.f);
        float* dst = tile + ((row >> 1) * DP + c4) * 2 + (row & 1);
        dst[0] = v.x; dst[2] = v.y; dst[4] = v.z; dst[6] = v.w;
      }
    }
    __syncthreads();
    for (int p = 0; p < pairs; ++p) {
      const float4* rp = reinterpret_cast<const float4*>(tile + p * (2 * DP));
      f32x2_t x[DP];
#pragma unroll
      for (int v = 0; v < DP / 2; ++v) { const float4 t = rp[v]; x[2 * v] = pk2f(t.x, t.y); x[2 * v + 1] = pk2f(t.z, t.w); }
      f32x2_t acc[kPairQpt];
#pragma unroll
      for (int r = 0; r < kPairQpt; ++r) acc[r] = x[DP - 1];             // |t|^2 of both rows
#pragma unroll
      for (int c = 0; c < DP - 1; ++c)
#pragma unroll
        for (int r = 0; r < kPairQpt; ++r) acc[r] = fma2f(qq[r][c], x[c], acc[r]);
#pragma unroll
      for (int r = 0; r < kPairQpt; ++r) {
        float s0, s1;
        unpk2f(acc[r], s0, s1);
        cand_insert<kKnnCand>(cd[r], ci[r], s0, (int)(base + 2 * p));
        cand_insert<kKnnCand>(cd[r], ci[r], s1, (int)(base + 2 * p + 1));
      }
    }
  }
#pragma unroll
  for (int r = 0; r < kPairQpt; ++r) {
    if (q0 + r < m) {
#pragma unroll
      for (int c = 0; c < kKnnCand; ++c) cand_idx[(q0 + r) * kKnnCand + c] = ci[r][c];
      cand_worst[q0 + r] = cd[r][kKnnCand - 1];
    }
  }
}

__device__ __forceinline__ double sqdist64(const double* q, const double* t, int d) {
  double s = 0.0;
  for (int j = 0; j < d; ++j) { const double x = q[j] - t[j]; s += x * x; }
  return s;
}

__device__ __forceinline__ bool less_di(double da, int64_t ia, double db, int64_t ib) {
  return da < db || (da == db && ia < ib);
}

// float64 rerank + certification.  One thread per query.
__global__ void knn_rerank_kernel(const double* __restrict__ train, const float* __restrict__ train32,
                                  int dp, int64_t n, const double* __restrict__ queries, int64_t m,
                                  int d, int k, int64_t index_base, const int32_t* __restrict__ labels,
                                  const int* __restrict__ cand_idx, const float* __restrict__ cand_worst,
                                  const float* __restrict__ qnorm, float tnorm_max, double err_rel, double err_floor,
                                  int64_t* __restrict__ nbr_idx, double* __restrict__ nbr_sqdist,
                                  int32_t* __restrict__ nbr_label, int32_t* __restrict__ redo_list,
                                  int32_t* __restrict__ redo_count, int32_t* __restrict__ refine_list,
                                  float* __restrict__ refine_thr, int refine_cap, float qnorm_limit,
                                  const double* __restrict__ bound, const float* __restrict__ thr0, bool allow_short) {
  const int64_t qi = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (qi >= m) return;
  const double* q = queries + qi * d;
  double cd[kKnnCand];
  int cidx[kKnnCand];
  int nc = 0;
  for (int c = 0; c < kKnnCand; ++c) {
    const int i = cand_idx[qi * kKnnCand + c];
    if (i < 0 || i >= n) continue;
    const double dd = sqdist64(q, train + (int64_t)i * d, d);
    int s = nc++;
    while (s > 0 && less_di(dd, i, cd[s - 1], cidx[s - 1])) { cd[s] = cd[s - 1]; cidx[s] = cidx[s - 1]; --s; }
    cd[s] = dd; cidx[s] = i;
  }
  const int kk = (int)min((int64_t)k, n);
  // a query outside the tensor-core filter's range was scored as the zero vector (knn_tc16_pack_kernel): its candidates
  // mean nothing -- exhaustive float64 scan
  const bool in_range = !(qnorm_limit > 0.f) || qnorm[qi] <= qnorm_limit;
  if (!in_range) nc = 0;
  // T = the radius inside which no row may be missing: the k-th exact candidate distance, and / or the caller's upper
  // bound U on the query's k-th distance (bounded calls: the shard is only asked for its rows within U, it may hold
  // fewer than k of them).  W = the score every row that is not a candidate is known to reach: the worst kept score once
  // the list has filled, and the threshold the filter started at.
  const double U = bound ? bound[qi] : INFINITY;
  const double Dk = nc >= kk ? cd[kk - 1] : INFINITY;
  const double T = fmin(Dk, U);
  // allow_short = false: the bound is the call's own (tile pruning), and k rows inside it are known to exist
  bool ok = in_range && T < INFINITY && (allow_short || nc >= kk);
  if (ok && (n > kKnnCand || bound)) {
    // The scan's score of row t is within err_rel * (|q| + |t|)^2 of |t|^2 - 2 q.t (the roundings act on terms bounded by
    // (|q| + |t|)^2).  A row that could still matter has exact distance <= T, hence |t| <= |q| + sqrt(T) by the triangle
    // inequality, hence score error <= err_rel * (2 |q| + sqrt(T))^2 -- the norm of the rows that matter, not of the
    // largest row of the train set (which made outliers in the train set reject 3 % of the queries of real feature
    // sets).  So: T < W + |q|^2 - err certifies that nothing inside the radius is missing.
    const float qn = qnorm[qi];
    const double brad = 2.0 * (double)sqrtf(qn) * 1.0000002 + sqrt(T);
    // err_floor: the split-fp16 filter also has an ABSOLUTE error (fp16 subnormal spacing of the lo planes), covered
    // by evaluating the relative bound at no less than err_floor
    const double err = err_rel * fmax(brad * brad, err_floor);
    const double W = fmin((double)cand_worst[qi], thr0 ? (double)thr0[qi] : INFINITY);
    ok = T < W + (double)qn - err;
  }
  if (!ok) {
    // Not certified.  Every row that can still matter has exact distance <= T, i.e. fp32 score <= T - |q|^2 + err32 -- the
    // threshold of the second pass (knn_refine_collect_kernel); without a refine list, without a radius, or past the
    // list's capacity: exhaustive float64 scan
    if (refine_list && in_range && T < INFINITY && train32) {
      const int slot = atomicAdd(redo_count + 1, 1);
      if (slot < refine_cap) {
        const float qn = qnorm[qi];
        const double brad = 2.0 * (double)sqrtf(qn) * 1.0000002 + sqrt(T);
        const double err32 = (double)(d + 4) * 1.1920929e-7 * brad * brad;
        refine_list[slot] = (int)qi;
        refine_thr[slot] = __double2float_ru(T - (double)qn + err32);
        return;
      }
    }
    const int slot = atomicAdd(redo_count, 1);
    redo_list[slot] = (int)qi;
    return;
  }
  const int have = min(kk, nc);
  for (int c = have; c < kk; ++c) {         // a bounded call whose shard holds fewer than k rows inside the radius
    if (nbr_idx) nbr_idx[qi * k + c] = -1;
    if (nbr_sqdist) nbr_sqdist[qi * k + c] = INFINITY;
    if (nbr_label) nbr_label[qi * k + c] = -1;
  }
  for (int c = 0; c < have; ++c) {
    if (nbr_idx) nbr_idx[qi * k + c] = index_base + cidx[c];
    if (nbr_sqdist) nbr_sqdist[qi * k + c] = cd[c];
    if (nbr_label) nbr_label[qi * k + c] = labels[cidx[c]];
  }
  for (int c = kk; c < k; ++c) {
    if (nbr_idx) nbr_idx[qi * k + c] = -1;
    if (nbr_sqdist) nbr_sqdist[qi * k + c] = INFINITY;
    if (nbr_label) nbr_label[qi * k + c] = -1;
  }
}

// The same rerank for wide feature vectors (the tensor-core path, D up to thousands): one WARP per query.  The
// query and its 8 candidate rows are read 32 features at a time by the whole warp (coalesced) into shared memory;
// lanes 0..7 each accumulate one candidate's distance over the features IN ORDER -- the very sum sqdist64 computes
// (products and sums round separately, -fmad=false), so certified and rescanned queries agree to the last bit.
constexpr int kRerankWarps = 8;
__global__ void __launch_bounds__(32 * kRerankWarps)
knn_rerank_wide_kernel(const double* __restrict__ train, int64_t n, const double* __restrict__ queries, int64_t m,
                       int d, int k, int64_t index_base, const int32_t* __restrict__ labels,
                       const int* __restrict__ cand_idx, const float* __restrict__ cand_worst,
                       const float* __restrict__ qnorm, float tnorm_max, double err_rel,
                       int64_t* __restrict__ nbr_idx, double* __restrict__ nbr_sqdist,
                       int32_t* __restrict__ nbr_label, int32_t* __restrict__ redo_list,
                       int32_t* __restrict__ redo_count) {
  __shared__ double stage[kRerankWarps][32][kKnnCand + 1];      // [feature][candidate | query]: conflict-free for lanes 0..7
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int64_t warps_total = (int64_t)gridDim.x * kRerankWarps;
  for (int64_t qi = (int64_t)blockIdx.x * kRerankWarps + w; qi < m; qi += warps_total) {
    const double* q = queries + qi * d;
    const int my_cand = lane < kKnnCand ? cand_idx[qi * kKnnCand + lane] : -1;
    double acc = 0.0;
    for (int c0 = 0; c0 < d; c0 += 32) {
      const int j = c0 + lane;
      stage[w][lane][kKnnCand] = j < d ? q[j] : 0.0;
#pragma unroll
      for (int c = 0; c < kKnnCand; ++c) {
        const int i = __shfl_sync(0xffffffffu, my_cand, c);
        stage[w][lane][c] = (i >= 0 && j < d) ? train[(int64_t)i * d + j] : 0.0;
      }
      __syncwarp();
      if (lane < kKnnCand) {
        const int lim = min(32, d - c0);
        for (int t = 0; t < lim; ++t) { const double x = stage[w][t][kKnnCand] - stage[w][t][lane]; acc += x * x; }
      }
      __syncwarp();
    }
    // lane 0 gathers the (distance, index) pairs and applies the certificate exactly like knn_rerank_kernel
    double cd[kKnnCand];
    int cidx[kKnnCand];
    int nc = 0;
#pragma unroll
    for (int c = 0; c < kKnnCand; ++c) {
      const double dd = __shfl_sync(0xffffffffu, acc, c);
      const int i = __shfl_sync(0xffffffffu, my_cand, c);
      if (i < 0) continue;
      int s = nc++;
      while (s > 0 && less_di(dd, i, cd[s - 1], cidx[s - 1])) { cd[s] = cd[s - 1]; cidx[s] = cidx[s - 1]; --s; }
      cd[s] = dd; cidx[s] = i;
    }
    if (lane != 0) continue;
    const int kk = (int)min((int64_t)k, n);
    bool ok = (nc >= kk);
    if (ok && n > kKnnCand) {
      const float qn = qnorm[qi];
      const double bound = (double)(sqrtf(qn) + sqrtf(tnorm_max));
      const double err = err_rel * bound * bound;
      const double lower = (double)cand_worst[qi] + (double)qn - err;
      ok = cd[kk - 1] < lower;
    }
    if (!ok) {
      const int slot = atomicAdd(redo_count, 1);
      redo_list[slot] = (int)qi;
      continue;
    }
    for (int c = 0; c < kk; ++c) {
      if (nbr_idx) nbr_idx[qi * k + c] = index_base + cidx[c];
      if (nbr_sqdist) nbr_sqdist[qi * k + c] = cd[c];
      if (nbr_label) nbr_label[qi * k + c] = labels[cidx[c]];
    }
    for (int c = kk; c < k; ++c) {
      if (nbr_idx) nbr_idx[qi * k + c] = -1;
      if (nbr_sqdist) nbr_sqdist[qi * k + c] = INFINITY;
      if (nbr_label) nbr_label[qi * k + c] = -1;
    }
  }
}

__host__ __device__ inline int rescan_parts(int grid, int total) { const int p = grid / (total > 0 ? total : 1); return p < 1 ? 1 : (p > 64 ? 64 : p); }

// Exhaustive float64 scan for the queries the certificate rejected: one warp per (query, slice of the train rows).
// A handful of rejected queries (the usual case: tens in a million) are split over up to 64 warps each -- partial
// lists to part_d / part_i, merged by knn_rescan_merge_kernel -- instead of leaving one warp to walk 10^5 rows
// (5 ms for 11 queries before the split); many rejected queries get one warp each and write their result directly.
__global__ void knn_rescan_kernel(const double* __restrict__ train, int64_t n,
                                  const double* __restrict__ queries, int d, int k, int64_t index_base,
                                  const int32_t* __restrict__ labels, const int32_t* __restrict__ redo_list,
                                  const int32_t* __restrict__ redo_count, int64_t* __restrict__ nbr_idx,
                                  double* __restrict__ nbr_sqdist, int32_t* __restrict__ nbr_label,
                                  double* __restrict__ part_d, long long* __restrict__ part_i) {
  const int lane = threadIdx.x & 31;
  const int warps_per_block = blockDim.x >> 5;
  const int total = *redo_count;
  if (total == 0) return;
  const int workers = gridDim.x * warps_per_block;
  const int parts = rescan_parts(workers, total);
  const int64_t rows_per = ((n + parts - 1) / parts + 31) / 32 * 32;
  for (int work = blockIdx.x * warps_per_block + (threadIdx.x >> 5); work < total * parts; work += workers) {
    const int item = work / parts, part = work % parts;
    const int64_t row_lo = (int64_t)part * rows_per, row_hi = min(n, row_lo + rows_per);
    const int64_t qi = redo_list[item];
    const double* q = queries + qi * d;
    double bd[kKnnMaxK];
    int64_t bi[kKnnMaxK];
    for (int c = 0; c < k; ++c) { bd[c] = INFINITY; bi[c] = INT64_MAX; }
    // 32 rows at a time: the warp copies their 32 * d contiguous doubles into shared memory with coalesced loads (a
    // lane walking its own row touches 32 different sectors per load: 6 ms for 100 rejected queries x 10^5 rows), then
    // every lane sums its row in feature order -- the very sum sqdist64 computes
    extern __shared__ double rescan_stage[];
    double* stage = rescan_stage + (size_t)(threadIdx.x >> 5) * 32 * d;
    for (int64_t i0 = row_lo; i0 < row_hi; i0 += 32) {
      const int rows = (int)min((int64_t)32, row_hi - i0);
      __syncwarp();
      for (int e = lane; e < rows * d; e += 32) stage[e] = train[i0 * d + e];
      __syncwarp();
      if (lane >= rows) continue;
      const int64_t i = i0 + lane;
      const double dd = sqdist64(q, stage + lane * d, d);
      if (less_di(dd, i, bd[k - 1], bi[k - 1])) {
        int s = k - 1;
        while (s > 0 && less_di(dd, i, bd[s - 1], bi[s - 1])) { bd[s] = bd[s - 1]; bi[s] = bi[s - 1]; --s; }
        bd[s] = dd; bi[s] = i;
      }
    }
    // merge the 32 sorted lists: k rounds of "global minimum, pop from its owner"
    int head = 0;
    for (int c = 0; c < k; ++c) {
      double md = head < k ? bd[head] : INFINITY;
      int64_t mi = head < k ? bi[head] : INT64_MAX;
      int owner = lane;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const double od = __shfl_xor_sync(0xffffffffu, md, o);
        const int64_t oi = __shfl_xor_sync(0xffffffffu, mi, o);
        const int oo = __shfl_xor_sync(0xffffffffu, owner, o);
        if (less_di(od, oi, md, mi)) { md = od; mi = oi; owner = oo; }
      }
      if (owner == lane && mi != INT64_MAX) ++head;
      if (lane == 0) {
        const bool valid = (mi != INT64_MAX);
        if (parts > 1) { part_d[(int64_t)work * kKnnMaxK + c] = valid ? md : INFINITY; part_i[(int64_t)work * kKnnMaxK + c] = mi; continue; }
        if (nbr_idx) nbr_idx[qi * k + c] = valid ? index_base + mi : -1;
        if (nbr_sqdist) nbr_sqdist[qi * k + c] = md;
        if (nbr_label) nbr_label[qi * k + c] = valid ? labels[mi] : -1;
      }
    }
  }
}

// The exhaustive float64 scan for wide feature vectors: one CTA (4 warps) per rejected query.  A warp takes 32 train
// rows at a time; the 32 x 32 block of features is read row by row (coalesced) into shared memory and every lane sums
// ITS row over the features in order -- the sum sqdist64 computes -- so the distances equal the other kernels' bit for bit.
constexpr int kRescanWarps = 4;
__global__ void __launch_bounds__(32 * kRescanWarps)
knn_rescan_wide_kernel(const double* __restrict__ train, int64_t n, const double* __restrict__ queries, int d, int k,
                       int64_t index_base, const int32_t* __restrict__ labels, const int32_t* __restrict__ redo_list,
                       const int32_t* __restrict__ redo_count, int64_t* __restrict__ nbr_idx,
                       double* __restrict__ nbr_sqdist, int32_t* __restrict__ nbr_label,
                       double* __restrict__ part_d, long long* __restrict__ part_i) {
  __shared__ double stage[kRescanWarps][32][33];            // [feature][row], padded: conflict-free both ways
  __shared__ double sq[kRescanWarps][32];
  __shared__ double m_d[kRescanWarps][kKnnMaxK];
  __shared__ long long m_i[kRescanWarps][kKnnMaxK];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int total = *redo_count;
  if (total == 0) return;
  // few rejected queries: the train rows of one query are split over `parts` CTAs (partial lists to part_d / part_i,
  // merged by knn_rescan_merge_kernel); many: one CTA per query writes the result itself
  const int parts = rescan_parts((int)gridDim.x, total);
  const int64_t rows_per = ((n + parts - 1) / parts + 32 * kRescanWarps - 1) / (32 * kRescanWarps) * (32 * kRescanWarps);
  for (int work = blockIdx.x; work < total * parts; work += gridDim.x) {
    const int item = work / parts, part = work % parts;
    const int64_t row_lo = (int64_t)part * rows_per, row_hi = min(n, row_lo + rows_per);
    const int64_t qi = redo_list[item];
    const double* q = queries + qi * d;
    double bd[kKnnMaxK];
    int64_t bi[kKnnMaxK];
    for (int c = 0; c < k; ++c) { bd[c] = INFINITY; bi[c] = INT64_MAX; }
    for (int64_t r0 = row_lo + (int64_t)w * 32; r0 < row_hi; r0 += 32 * kRescanWarps) {
      const int64_t i = r0 + lane;
      double acc = 0.0;
      for (int c0 = 0; c0 < d; c0 += 32) {
        const int j = c0 + lane;
        sq[w][lane] = j < d ? q[j] : 0.0;
        for (int rr = 0; rr < 32; ++rr)
          stage[w][lane][rr] = (r0 + rr < row_hi && j < d) ? train[(r0 + rr) * d + j] : 0.0;
        __syncwarp();
        const int lim = min(32, d - c0);
        for (int t = 0; t < lim; ++t) { const double x = sq[w][t] - stage[w][t][lane]; acc += x * x; }
        __syncwarp();
      }
      if (i < row_hi && less_di(acc, i, bd[k - 1], bi[k - 1])) {
        int s = k - 1;
        while (s > 0 && less_di(acc, i, bd[s - 1], bi[s - 1])) { bd[s] = bd[s - 1]; bi[s] = bi[s - 1]; --s; }
        bd[s] = acc; bi[s] = i;
      }
    }
    // merge the warp's 32 sorted lists (k rounds of "global minimum, pop from its owner") into shared memory
    int head = 0;
    for (int c = 0; c < k; ++c) {
      double md = head < k ? bd[head] : INFINITY;
      int64_t mi = head < k ? bi[head] : INT64_MAX;
      int owner = lane;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const double od = __shfl_xor_sync(0xffffffffu, md, o);
        const int64_t oi = __shfl_xor_sync(0xffffffffu, mi, o);
        const int oo = __shfl_xor_sync(0xffffffffu, owner, o);
        if (less_di(od, oi, md, mi)) { md = od; mi = oi; owner = oo; }
      }
      if (owner == lane && mi != INT64_MAX) ++head;
      if (lane == 0) { m_d[w][c] = md; m_i[w][c] = mi; }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      int hp[kRescanWarps] = {0, 0, 0, 0};
      for (int c = 0; c < k; ++c) {
        int best = -1;
        for (int ww = 0; ww < kRescanWarps; ++ww)
          if (hp[ww] < k && (best < 0 || less_di(m_d[ww][hp[ww]], m_i[ww][hp[ww]], m_d[best][hp[best]], m_i[best][hp[best]]))) best = ww;
        const double md = best >= 0 ? m_d[best][hp[best]] : INFINITY;
        const int64_t mi = best >= 0 ? (int64_t)m_i[best][hp[best]] : INT64_MAX;
        if (best >= 0) ++hp[best];
        const bool valid = (mi != INT64_MAX);
        if (parts > 1) { part_d[(int64_t)work * kKnnMaxK + c] = valid ? md : INFINITY; part_i[(int64_t)work * kKnnMaxK + c] = mi; continue; }
        if (nbr_idx) nbr_idx[qi * k + c] = valid ? index_base + mi : -1;
        if (nbr_sqdist) nbr_sqdist[qi * k + c] = valid ? md : INFINITY;
        if (nbr_label) nbr_label[qi * k + c] = valid ? labels[mi] : -1;
      }
    }
    __syncthreads();
  }
}

// merge of the per-part lists of knn_rescan_wide_kernel: one thread per rejected query
__global__ void knn_rescan_merge_kernel(int grid_of_scan, int k, int64_t index_base, const int32_t* __restrict__ labels,
                                        const int32_t* __restrict__ redo_list, const int32_t* __restrict__ redo_count,
                                        const double* __restrict__ part_d, const long long* __restrict__ part_i,
                                        int64_t* __restrict__ nbr_idx, double* __restrict__ nbr_sqdist,
                                        int32_t* __restrict__ nbr_label) {
  const int total = *redo_count;
  if (total == 0) return;
  const int parts = rescan_parts(grid_of_scan, total);
  if (parts == 1) return;
  const int item = blockIdx.x * blockDim.x + threadIdx.x;
  if (item >= total) return;
  const int64_t qi = redo_list[item];
  int hp[64];
  for (int p = 0; p < parts; ++p) hp[p] = 0;
  for (int c = 0; c < k; ++c) {
    int best = -1;
    double bdv = INFINITY; long long biv = INT64_MAX;
    for (int p = 0; p < parts; ++p) {
      if (hp[p] >= k) continue;
      const int64_t o = ((int64_t)item * parts + p) * kKnnMaxK + hp[p];
      const double dv = part_d[o]; const long long iv = part_i[o];
      if (iv != INT64_MAX && (best < 0 || less_di(dv, iv, bdv, biv))) { best = p; bdv = dv; biv = iv; }
    }
    if (best >= 0) ++hp[best];
    const bool valid = best >= 0;
    if (nbr_idx) nbr_idx[qi * k + c] = valid ? index_base + biv : -1;
    if (nbr_sqdist) nbr_sqdist[qi * k + c] = valid ? bdv : INFINITY;
    if (nbr_label) nbr_label[qi * k + c] = valid ? labels[biv] : -1;
  }
}

// train float64 [n,d] -> padded fp32 rows with |t|^2 in the last column; also max |t|^2.
__global__ void knn_pack_kernel(const double* __restrict__ train, int64_t n, int d, int dp,
                                float* __restrict__ train32, float* __restrict__ tnorm_max) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  float nn = 0.f;
  if (i < n) {
    for (int j = 0; j < dp - 1; ++j) {
      const float v = j < d ? (float)train[i * d + j] : 0.f;
      train32[i * dp + j] = v;
      nn = fmaf(v, v, nn);
    }
    train32[i * dp + dp - 1] = nn;
  }
  nn = warp_reduce(nn, [](float a, float b) { return fmaxf(a, b); });
  if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<int*>(tnorm_max), __float_as_int(nn));
}

// majority vote over k neighbour labels, ties to the smallest label
// (sklearn/neighbors/_classification.py:262-309); one thread per query.
__global__ void knn_vote_kernel(const int32_t* __restrict__ nbr_label, int64_t m, int k,
                                int32_t* __restrict__ out) {
  const int64_t qi = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (qi >= m) return;
  const int32_t* l = nbr_label + qi * k;
  int best = -1, best_cnt = 0;
  for (int a = 0; a < k; ++a) {
    if (l[a] < 0) continue;
    int cnt = 0;
    for (int b = 0; b < k; ++b) cnt += (l[b] == l[a]);
    if (cnt > best_cnt || (cnt == best_cnt && l[a] < best)) { best = l[a]; best_cnt = cnt; }
  }
  out[qi] = best;
}

// merge R candidate lists [R, m, k] -> global top-k by (distance, index), then vote.
__global__ void knn_merge_vote_kernel(const double* __restrict__ cd, const int64_t* __restrict__ ci,
                                      const int32_t* __restrict__ cl, int r, int64_t m, int k,
                                      int32_t* __restrict__ labels_out, int64_t* __restrict__ idx_out,
                                      double* __restrict__ dist_out) {
  const int64_t qi = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (qi >= m) return;
  double bd[kKnnMaxK];
  int64_t bi[kKnnMaxK];
  int32_t bl[kKnnMaxK];
  for (int c = 0; c < k; ++c) { bd[c] = INFINITY; bi[c] = INT64_MAX; bl[c] = -1; }
  for (int s = 0; s < r; ++s) {
    for (int c = 0; c < k; ++c) {
      const int64_t o = ((int64_t)s * m + qi) * k + c;
      const int64_t idx = ci[o];
      if (idx < 0) continue;
      const double dd = cd[o];
      if (less_di(dd, idx, bd[k - 1], bi[k - 1])) {
        int p = k - 1;
        while (p > 0 && less_di(dd, idx, bd[p - 1], bi[p - 1])) { bd[p] = bd[p - 1]; bi[p] = bi[p - 1]; bl[p] = bl[p - 1]; --p; }
        bd[p] = dd; bi[p] = idx; bl[p] = cl[o];
      }
    }
  }
  int best = -1, best_cnt = 0;
  for (int a = 0; a < k; ++a) {
    if (bl[a] < 0) continue;
    int cnt = 0;
    for (int b = 0; b < k; ++b) cnt += (bl[b] == bl[a]);
    if (cnt > best_cnt || (cnt == best_cnt && bl[a] < best)) { best = bl[a]; best_cnt = cnt; }
  }
  if (labels_out) labels_out[qi] = best;
  for (int c = 0; c < k; ++c) {
    if (idx_out) idx_out[qi * k + c] = bi[c] == INT64_MAX ? -1 : bi[c];
    if (dist_out) dist_out[qi * k + c] = bd[c];
  }
}

__global__ void knn_iota_kernel(int32_t* list, int32_t* count, int64_t m) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < m) list[i] = (int32_t)i;
  if (i == 0) { count[0] = (int32_t)m; count[1] = 0; count[2] = 0; }
}


// ---------------------------------------------------------------------------------------
// Second pass for the queries the certificate rejected (D <= 15 path): instead of an exhaustive float64 scan per query
// (the 12 MB train matrix through L2 once per rejected query), score every row again in fp32 against the query's OWN
// threshold -- rows whose score is above it cannot be among the k nearest (rerank kernel) -- and keep the survivors
// (typically a dozen); knn_refine_finish_kernel ranks those in float64 exactly as the rescan would.  A query with
// more than kRefineCap survivors goes to the exhaustive scan.  Work items = (block of 128 rejected queries) x (part of
// the train rows), persistent grid, everything sized on the device: no host round trip.
// ---------------------------------------------------------------------------------------
__global__ void knn_bound_thresholds_kernel(const double* __restrict__ bound, const float* __restrict__ qnorm, int64_t m,
                                            double err_rel, double err_floor, float* __restrict__ thr0) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= m) return;
  const double U = bound[i];
  float t = INFINITY;
  if (U < INFINITY && U >= 0.0) {
    const double qn = (double)qnorm[i];
    const double brad = 2.0 * sqrt(qn) * 1.0000002 + sqrt(U);
    const double err = err_rel * fmax(brad * brad, err_floor);
    // twice the error: once for the rows' scores, once so that the rerank certificate (strict) holds at T = U
    t = __double2float_ru((U - qn + 2.0 * err) * (U - qn + 2.0 * err >= 0.0 ? 1.000001 : 0.999999));
  }
  thr0[i] = t;
}

constexpr int kRefineCap = 64;
constexpr int kRefineThreads = 128;

template <int DP>
__global__ void __launch_bounds__(kRefineThreads)
knn_refine_collect_kernel(const float* __restrict__ train32, int64_t n, const double* __restrict__ queries, int d,
                          const int32_t* __restrict__ refine_list, const float* __restrict__ refine_thr,
                          const int32_t* __restrict__ counts, int refine_cap, int32_t* __restrict__ surv_count,
                          int32_t* __restrict__ surv_rows) {
  __shared__ __align__(16) float tile[kTileRows * DP];
  const int total = min(counts[1], refine_cap);
  if (total == 0) return;
  const int qblocks = (total + kRefineThreads - 1) / kRefineThreads;
  int parts = (int)gridDim.x / qblocks;
  if (parts < 1) parts = 1;
  const int64_t tiles = (n + kTileRows - 1) / kTileRows;
  if (parts > tiles) parts = (int)tiles;
  const int64_t tiles_per = (tiles + parts - 1) / parts;
  for (int work = blockIdx.x; work < qblocks * parts; work += gridDim.x) {
    const int qb = work / parts, part = work % parts;
    const int slot = qb * kRefineThreads + threadIdx.x;
    const bool live = slot < total;
    float q[DP - 1];
    float thr = -INFINITY;
    if (live) {
      const int64_t qi = refine_list[slot];
      thr = refine_thr[slot];
#pragma unroll
      for (int j = 0; j < DP - 1; ++j) q[j] = j < d ? -2.f * (float)queries[qi * d + j] : 0.f;
    } else {
#pragma unroll
      for (int j = 0; j < DP - 1; ++j) q[j] = 0.f;
    }
    const int64_t row_lo = (int64_t)part * tiles_per * kTileRows, row_hi = min(n, row_lo + tiles_per * kTileRows);
    for (int64_t base = row_lo; base < row_hi; base += kTileRows) {
      const int rows = (int)min((int64_t)kTileRows, row_hi - base);
      __syncthreads();
      {
        const float4* src = reinterpret_cast<const float4*>(train32 + base * DP);
        float4* dst = reinterpret_cast<float4*>(tile);
        for (int i = threadIdx.x; i < rows * (DP / 4); i += kRefineThreads) dst[i] = src[i];
      }
      __syncthreads();
      for (int j = 0; j < rows; ++j) {
        const float4* row = reinterpret_cast<const float4*>(tile + j * DP);
        float acc = tile[j * DP + DP - 1];
#pragma unroll
        for (int v = 0; v < DP / 4; ++v) {
          const float4 x = row[v];
          acc = fmaf(q[4 * v], x.x, acc);
          acc = fmaf(q[4 * v + 1], x.y, acc);
          acc = fmaf(q[4 * v + 2], x.z, acc);
          if (4 * v + 3 < DP - 1) acc = fmaf(q[4 * v + 3], x.w, acc);
        }
        if (acc <= thr) {
          const int s = atomicAdd(surv_count + slot, 1);
          if (s < kRefineCap) surv_rows[(int64_t)slot * kRefineCap + s] = (int)(base + j);
        }
      }
    }
  }
}

// one warp per rejected query: float64 distances of its survivors, the k smallest by (distance, index)
__global__ void knn_refine_finish_kernel(const double* __restrict__ train, const double* __restrict__ queries, int d, int k,
                                         int64_t index_base, const int32_t* __restrict__ labels,
                                         const int32_t* __restrict__ refine_list, int32_t* __restrict__ counts, int refine_cap,
                                         const int32_t* __restrict__ surv_count, const int32_t* __restrict__ surv_rows,
                                         int64_t* __restrict__ nbr_idx, double* __restrict__ nbr_sqdist,
                                         int32_t* __restrict__ nbr_label, int32_t* __restrict__ redo_list, bool allow_short) {
  const int lane = threadIdx.x & 31;
  const int total = min(counts[1], refine_cap);
  const int warps = (gridDim.x * blockDim.x) >> 5;
  for (int slot = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; slot < total; slot += warps) {
    const int64_t qi = refine_list[slot];
    const int cnt = surv_count[slot];
    if (cnt > kRefineCap || (cnt < k && !allow_short)) {       // too many survivors (or, in an unbounded call, too few): exhaustive float64 scan
      if (lane == 0) { const int s = atomicAdd(counts, 1); redo_list[s] = (int)qi; atomicAdd(counts + 2, 1); }
      continue;
    }
    const double* q = queries + qi * d;
    double dd[kRefineCap / 32];
    int64_t ii[kRefineCap / 32];
#pragma unroll
    for (int r = 0; r < kRefineCap / 32; ++r) {
      const int e = lane + 32 * r;
      dd[r] = INFINITY; ii[r] = INT64_MAX;
      if (e < cnt) { ii[r] = surv_rows[(int64_t)slot * kRefineCap + e]; dd[r] = sqdist64(q, train + ii[r] * d, d); }
    }
    for (int c = 0; c < k; ++c) {
      // the lane's smallest remaining entry, then the warp's
      int br = 0;
#pragma unroll
      for (int r = 1; r < kRefineCap / 32; ++r) if (less_di(dd[r], ii[r], dd[br], ii[br])) br = r;
      double md = dd[0]; int64_t mi = ii[0];
#pragma unroll
      for (int r = 1; r < kRefineCap / 32; ++r) if (br == r) { md = dd[r]; mi = ii[r]; }
      int owner = lane;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const double od = __shfl_xor_sync(0xffffffffu, md, o);
        const int64_t oi = __shfl_xor_sync(0xffffffffu, mi, o);
        const int oo = __shfl_xor_sync(0xffffffffu, owner, o);
        if (less_di(od, oi, md, mi)) { md = od; mi = oi; owner = oo; }
      }
      if (owner == lane) {
#pragma unroll
        for (int r = 0; r < kRefineCap / 32; ++r) if (br == r) { dd[r] = INFINITY; ii[r] = INT64_MAX; }
      }
      if (lane == 0) {
        const bool valid = mi != INT64_MAX;           // bounded calls: fewer than k rows inside the radius
        if (nbr_idx) nbr_idx[qi * k + c] = valid ? index_base + mi : -1;
        if (nbr_sqdist) nbr_sqdist[qi * k + c] = md;
        if (nbr_label) nbr_label[qi * k + c] = valid ? labels[mi] : -1;
      }
    }
  }
}

}  // namespace

int knn_rescan_grid(int sm_count) { return sm_count * 16; }      // work items of either rescan kernel (narrow: 2 blocks x 8 warps per SM)

int knn_padded_dim(int d) {
  if (d + 1 <= 16) return 16;
  if (d + 1 <= 32) return 32;
  if (d + 1 <= 64) return 64;
  return 0;
}

cudaError_t knn_pack(const double* train, int64_t n, int d, int dp, float* train32, float* tnorm_max,
                     cudaStream_t st) {
  cudaMemsetAsync(tnorm_max, 0, sizeof(float), st);
  if (n > 0) knn_pack_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(train, n, d, dp, train32, tnorm_max);
  return cudaGetLastError();
}

cudaError_t knn_scan(int dp, const float* train32, int64_t n, const double* q, int64_t m, int d,
                     int* cand_idx, float* cand_worst, float* qnorm, cudaStream_t st) {
  if (m == 0) return cudaSuccess;
  if (dp == 16) {
    constexpr int QPT = 2;
    const unsigned grid = (unsigned)((m + (int64_t)kScanThreads * QPT - 1) / ((int64_t)kScanThreads * QPT));
    knn_scan_pair_kernel<<<grid, kScanThreads, 0, st>>>(train32, n, q, m, d, cand_idx, cand_worst, qnorm);
  } else if (dp == 32) {
    const unsigned grid = (unsigned)((m + kScanThreads - 1) / kScanThreads);
    knn_scan_kernel<32, 1><<<grid, kScanThreads, 0, st>>>(train32, n, q, m, d, cand_idx, cand_worst, qnorm);
  } else {
    const unsigned grid = (unsigned)((m + kScanThreads - 1) / kScanThreads);
    knn_scan_kernel<64, 1><<<grid, kScanThreads, 0, st>>>(train32, n, q, m, d, cand_idx, cand_worst, qnorm);
  }
  return cudaGetLastError();
}

cudaError_t knn_rerank(const double* train, const float* train32, int dp, int64_t n, const double* q,
                       int64_t m, int d, int k, int64_t index_base, const int32_t* labels,
                       const int* cand_idx, const float* cand_worst, const float* qnorm,
                       float tnorm_max_host, double err_rel, double err_floor, int64_t* nbr_idx, double* nbr_sqdist, int32_t* nbr_label,
                       int32_t* redo_list, int32_t* redo_count, cudaStream_t st, int32_t* refine_list, float* refine_thr,
                       int refine_cap, float qnorm_limit, const double* bound, const float* thr0, bool allow_short) {
  if (m == 0) return cudaSuccess;
  cudaMemsetAsync(redo_count, 0, 4 * sizeof(int32_t), st);
  if (d > 64) {
    const unsigned grid = (unsigned)std::min<int64_t>((m + kRerankWarps - 1) / kRerankWarps, 148 * 32);
    knn_rerank_wide_kernel<<<grid, 32 * kRerankWarps, 0, st>>>(train, n, q, m, d, k, index_base, labels, cand_idx, cand_worst, qnorm,
                                                                tnorm_max_host, err_rel, nbr_idx, nbr_sqdist, nbr_label, redo_list,
                                                                redo_count);
    return cudaGetLastError();
  }
  knn_rerank_kernel<<<(unsigned)((m + 127) / 128), 128, 0, st>>>(
      train, train32, dp, n, q, m, d, k, index_base, labels, cand_idx, cand_worst, qnorm, tnorm_max_host, err_rel, err_floor,
      nbr_idx, nbr_sqdist, nbr_label, redo_list, redo_count, refine_list, refine_thr, refine_cap, qnorm_limit, bound, thr0,
      allow_short);
  return cudaGetLastError();
}

int knn_refine_survivor_cap() { return kRefineCap; }

cudaError_t knn_bound_thresholds(const double* bound, const float* qnorm, int64_t m, double err_rel, double err_floor, float* thr0,
                                 cudaStream_t st) {
  if (m == 0) return cudaSuccess;
  knn_bound_thresholds_kernel<<<(unsigned)((m + 255) / 256), 256, 0, st>>>(bound, qnorm, m, err_rel, err_floor, thr0);
  return cudaGetLastError();
}

cudaError_t knn_refine(const double* train, const float* train32, int dp, int64_t n, const double* q, int d, int k,
                       int64_t index_base, const int32_t* labels, const int32_t* refine_list, const float* refine_thr,
                       int refine_cap, int32_t* surv_count, int32_t* surv_rows, int32_t* counts, int32_t* redo_list,
                       int64_t* nbr_idx, double* nbr_sqdist, int32_t* nbr_label, int sm_count, cudaStream_t st, bool allow_short) {
  if (dp != 16 || refine_cap <= 0) return cudaSuccess;
  cudaMemsetAsync(surv_count, 0, sizeof(int32_t) * (size_t)refine_cap, st);
  knn_refine_collect_kernel<16><<<sm_count * 4, kRefineThreads, 0, st>>>(train32, n, q, d, refine_list, refine_thr, counts, refine_cap,
                                                                          surv_count, surv_rows);
  knn_refine_finish_kernel<<<sm_count * 2, 256, 0, st>>>(train, q, d, k, index_base, labels, refine_list, counts, refine_cap,
                                                          surv_count, surv_rows, nbr_idx, nbr_sqdist, nbr_label, redo_list, allow_short);
  return cudaGetLastError();
}

cudaError_t knn_redo_all(int32_t* redo_list, int32_t* redo_count, int64_t m, cudaStream_t st) {
  if (m == 0) return cudaSuccess;
  knn_iota_kernel<<<(unsigned)((m + 255) / 256), 256, 0, st>>>(redo_list, redo_count, m);
  return cudaGetLastError();
}

cudaError_t knn_rescan(const double* train, int64_t n, const double* q, int d, int k, int64_t index_base,
                       const int32_t* labels, const int32_t* redo_list, const int32_t* redo_count,
                       int64_t* nbr_idx, double* nbr_sqdist, int32_t* nbr_label, int sm_count,
                       double* part_d, long long* part_i, int max_redo, cudaStream_t st) {
  if (d > 64) {
    const int grid = knn_rescan_grid(sm_count);
    knn_rescan_wide_kernel<<<grid, 32 * kRescanWarps, 0, st>>>(train, n, q, d, k, index_base, labels, redo_list,
                                                               redo_count, nbr_idx, nbr_sqdist, nbr_label, part_d, part_i);
    // parts > 1 only when fewer than `grid` queries were rejected: that many merge threads are enough
    const int mt = max_redo < grid ? max_redo : grid;
    if (mt > 0)
      knn_rescan_merge_kernel<<<(mt + 127) / 128, 128, 0, st>>>(grid, k, index_base, labels, redo_list, redo_count, part_d, part_i,
                                                               nbr_idx, nbr_sqdist, nbr_label);
  } else {
    const int blocks = sm_count * 2, workers = blocks * 8;          // knn_rescan_grid(sm_count) >= workers: the partial lists fit
    const size_t stage_bytes = (size_t)8 * 32 * d * sizeof(double);      // d <= 64: at most 128 KB
    cudaError_t ea = cudaFuncSetAttribute(knn_rescan_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)stage_bytes);
    if (ea != cudaSuccess) return ea;
    knn_rescan_kernel<<<blocks, 256, stage_bytes, st>>>(train, n, q, d, k, index_base, labels, redo_list, redo_count, nbr_idx, nbr_sqdist,
                                                        nbr_label, part_d, part_i);
    const int mt = max_redo < workers ? max_redo : workers;
    if (mt > 0)
      knn_rescan_merge_kernel<<<(mt + 127) / 128, 128, 0, st>>>(workers, k, index_base, labels, redo_list, redo_count, part_d, part_i,
                                                               nbr_idx, nbr_sqdist, nbr_label);
  }
  return cudaGetLastError();
}

cudaError_t knn_vote(const int32_t* nbr_label, int64_t m, int k, int32_t* out, cudaStream_t st) {
  if (m == 0) return cudaSuccess;
  knn_vote_kernel<<<(unsigned)((m + 255) / 256), 256, 0, st>>>(nbr_label, m, k, out);
  return cudaGetLastError();
}

cudaError_t knn_merge_vote(const double* cd, const int64_t* ci, const int32_t* cl, int r, int64_t m,
                           int k, int32_t* labels_out, int64_t* idx_out, double* dist_out,
                           cudaStream_t st) {
  if (m == 0) return cudaSuccess;
  knn_merge_vote_kernel<<<(unsigned)((m + 255) / 256), 256, 0, st>>>(cd, ci, cl, r, m, k, labels_out,
                                                                    idx_out, dist_out);
  return cudaGetLastError();
}

}  // namespace dsp
