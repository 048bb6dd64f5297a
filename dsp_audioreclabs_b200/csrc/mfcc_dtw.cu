// MFCC + DTW template matching (BASELINE config 5, SURVEY.md section 8 rows a11 / f4).
//
// NOT present in the reference (no mfcc / dtw / fft anywhere under /root/reference): the definition is the
// textbook one written down in oracle/mfcc_dtw_oracle.py ("self-oracle, parity unpinned"), built on the reference's
// own pre-processing (src/audio_processing.py:49-90), endpoints (:135-275) and framing rule (:299-333).
//
//   mfcc_kernel   one CTA per utterance (persistent over a work counter): DC / peak of the utterance from exact integer
//                 sums, then per frame of the trimmed segment: pre-emphasis + window -> radix-2 FFT in shared memory ->
//                 power spectrum -> mel filterbank (one warp per filter over its non-zero bins) -> log -> DCT-II.
//                 Filterbank, DCT matrix, twiddles and window are caller-provided tables: the kernel fixes no constants.
//   dtw_kernel    one 32-thread CTA per (query, template) pair, anti-diagonal wavefront: lane L owns a strip of R
//                 consecutive query frames and runs one column behind lane L-1; the boundary value D[i-1][j] travels
//                 by one shuffle per step, template frames are read from shared memory (stride 13 floats: conflict
//                 free), query frames live in registers.  Cost matrix [queries x templates] in fp32.
//   dtw_topk      one warp per query: the k smallest costs (ties to the lower template index) -> candidates in the
//                 layout knn_merge_vote consumes, so the row-sharded multi-GPU exchange is the KNN one.
//   dtw_topk_fused  the same top k without the cost matrix: one warp per (query, slice of templates) keeps the slice's k
//                 best in registers and abandons a pair once a lower bound on its cost exceeds the k-th;
//                 dtw_merge_kernel combines the slices with dtw_topk's selection.  Same cell arithmetic
//                 (dtw_lane_column), so the same bits as the matrix path.
#include <algorithm>
#include <cfloat>
#include <type_traits>

#include <climits>
#include "kernels.cuh"
#include "knn.cuh"
#include "mfcc_dtw.cuh"

namespace dsp {

namespace {

constexpr int kMfccThreads = 256;

__device__ __forceinline__ long long block_sum_ll(long long v, long long* sh) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if (lane == 0) sh[w] = v;
  __syncthreads();
  long long t = 0;
  for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t += sh[i];
  __syncthreads();
  return t;
}
__device__ __forceinline__ int block_min_i(int v, int* sh) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  v = __reduce_min_sync(0xffffffffu, v);
  if (lane == 0) sh[w] = v;
  __syncthreads();
  int t = sh[0];
  for (int i = 1; i < (int)(blockDim.x >> 5); ++i) t = min(t, sh[i]);
  __syncthreads();
  return t;
}

__global__ void __launch_bounds__(kMfccThreads)
mfcc_kernel(const int16_t* __restrict__ samples, const int64_t* __restrict__ offsets, const int32_t* __restrict__ lengths,
            const int32_t* __restrict__ seg_start, const int32_t* __restrict__ seg_end, int64_t n_utts, MfccArgs a,
            const float* __restrict__ window, const float2* __restrict__ twiddle, const float* __restrict__ filterbank,
            const int2* __restrict__ fb_range, const float* __restrict__ dct, const int64_t* __restrict__ mfcc_offsets,
            float* __restrict__ out, int32_t* __restrict__ n_frames_out, unsigned int* __restrict__ work_counter) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float2* buf = reinterpret_cast<float2*>(smem_raw);                       // n_fft complex values
  float* power = reinterpret_cast<float*>(buf + a.n_fft);                  // n_fft / 2 + 1
  float* logmel = power + (a.n_fft / 2 + 1);                               // n_mels
  __shared__ long long sh_ll[kMfccThreads / 32];
  __shared__ int sh_i[kMfccThreads / 32];
  __shared__ unsigned int sh_u;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int n_fft = a.n_fft, half_fft = n_fft >> 1, n_bins = half_fft + 1;
  const int log2n = 31 - __clz(n_fft);
  for (;;) {
    if (tid == 0) sh_u = atomicAdd(work_counter, 1u);
    __syncthreads();
    const int64_t u = sh_u;
    __syncthreads();
    if (u >= n_utts) break;
    const int16_t* x = samples + offsets[u];
    const int n = lengths ? lengths[u] : (int)(offsets[u + 1] - offsets[u]);
    // ---- remove_dc + normalize_audio constants (src/audio_processing.py:49-75) from exact integer sums
    long long s = 0; int mn = 32767, mx = -32768;
    for (int i = tid; i < n; i += kMfccThreads) { const int k = x[i]; s += k; mn = min(mn, k); mx = max(mx, k); }
    const long long S = block_sum_ll(s, sh_ll);
    mn = block_min_i(mn, sh_i);
    mx = -block_min_i(-mx, sh_i);
    const long long N = n > 0 ? n : 1;
    const long long M = max(N * mx - S, S - N * mn);                      // N * max|k - mean|
    const double mu = (double)S / (double)N;
    const double scale = M > 0 ? (double)N / (double)M : 1.0 / 32768.0;   // all samples equal: x - mean = 0 anyway
    const int start = seg_start[u], end = min(seg_end[u], n);
    const int seg = end - start;
    // rows [mfcc_offsets[u], mfcc_offsets[u + 1]) belong to the utterance: never more frames than that capacity
    const int nf = (int)std::min<int64_t>(frame_count_host_device(seg, a.frame_length, a.frame_shift), mfcc_offsets[u + 1] - mfcc_offsets[u]);
    if (tid == 0 && n_frames_out) n_frames_out[u] = nf;
    const int64_t obase = mfcc_offsets[u];
    for (int f = 0; f < nf; ++f) {
      const int p = start + f * a.frame_shift;
      const int valid = min(a.frame_length, end - p);
      // ---- pre-emphasis + window, stored in bit-reversed order for the in-place decimation-in-time FFT
      for (int j = tid; j < n_fft; j += kMfccThreads) {
        float v = 0.f;
        if (j < valid) {
          const double cur = ((double)x[p + j] - mu) * scale;
          const double prv = (p + j > start) ? ((double)x[p + j - 1] - mu) * scale : 0.0;
          v = (float)(cur - a.pre_emphasis * prv) * window[j];
        }
        buf[__brev((unsigned)j) >> (32 - log2n)] = make_float2(v, 0.f);
      }
      __syncthreads();
      for (int st = 1; st <= log2n; ++st) {
        const int half = 1 << (st - 1);
        const int tw_stride = half_fft >> (st - 1);
        for (int b = tid; b < half_fft; b += kMfccThreads) {
          const int pos = b & (half - 1);
          const int i0 = ((b >> (st - 1)) << st) + pos, i1 = i0 + half;
          const float2 w = __ldg(twiddle + pos * tw_stride);
          const float2 lo = buf[i0], hi = buf[i1];
          const float tr = hi.x * w.x - hi.y * w.y, ti = hi.x * w.y + hi.y * w.x;
          buf[i0] = make_float2(lo.x + tr, lo.y + ti);
          buf[i1] = make_float2(lo.x - tr, lo.y - ti);
        }
        __syncthreads();
      }
      const float inv_nfft = 1.0f / (float)n_fft;
      for (int b = tid; b < n_bins; b += kMfccThreads) { const float2 c = buf[b]; power[b] = (c.x * c.x + c.y * c.y) * inv_nfft; }
      __syncthreads();
      // ---- mel filterbank: one warp per filter over its non-zero bins
      for (int m = wid; m < a.n_mels; m += kMfccThreads / 32) {
        const int2 r = fb_range[m];
        float acc = 0.f;
        for (int b = r.x + lane; b < r.y; b += 32) acc = fmaf(__ldg(filterbank + (size_t)m * n_bins + b), power[b], acc);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == 0) logmel[m] = logf(fmaxf(acc, a.log_floor));
      }
      __syncthreads();
      // ---- DCT-II
      for (int c = tid; c < a.n_ceps; c += kMfccThreads) {
        float acc = 0.f;
        for (int m = 0; m < a.n_mels; ++m) acc = fmaf(__ldg(dct + c * a.n_mels + m), logmel[m], acc);
        out[(obase + f) * a.n_ceps + c] = acc;
      }
      __syncthreads();
    }
  }
}

// ---------------------------------------------------------------------------------------
// DTW: one warp per (query, template) pair
// ---------------------------------------------------------------------------------------
// Lane L owns R consecutive query frames of a STRIP of 32 R rows (in registers) and runs one column behind lane L - 1:
// D[i-1][j] crosses the lane boundary by one shfl_up per step.  Queries longer than a strip are processed strip by
// strip: the strip's last row is kept in shared memory (one float per template frame, written in place -- lane 0 has
// read column j long before the last lane overwrites it) and enters the next strip as its top boundary.  DMAX bounds
// the feature dimension held in registers (R * DMAX <= 128 floats per lane): 16 for the 13 MFCCs, 32 / 64 / 128 for
// stacked delta features or other embeddings.
constexpr int kDtwMaxDim = 128;
constexpr int kDtwFusedWarps = 4;               // warps per CTA of dtw_topk_fused_kernel (fewer when shared memory is short)

// The R cells a lane owns in column j: D[i][j] = |q_i - t_j| + min(D[i-1][j], D[i][j-1], D[i-1][j-1]).  The one
// definition of the cell arithmetic (fmaf order, sqrtf, fminf nesting) behind every DTW cost this library reports, so
// the cost-matrix and the fused top-k paths agree bit for bit.  up / diag: D[i-1][j] / D[i-1][j-1] of the lane's first
// row; prev: D[i][j-1] of its rows, replaced by D[i][j].  Returns min_r D[i][j] over the lane's rows.
template <int R, int DMAX>
__device__ __forceinline__ float dtw_lane_column(const float (&q)[R][DMAX], const float* __restrict__ tj, int dim, int i_lane,
                                                 int n, int i_last, int j, float up, float diag, float (&prev)[R], float& cur_r) {
  float t[DMAX];
#pragma unroll
  for (int c = 0; c < DMAX; ++c) t[c] = c < dim ? tj[c] : 0.f;
  float row_min = INFINITY;
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int i = i_lane + r;
    float d2 = 0.f;
#pragma unroll
    for (int c = 0; c < DMAX; ++c) { const float e = q[r][c] - t[c]; d2 = fmaf(e, e, d2); }
    const float d = sqrtf(d2);
    float best = fminf(fminf(up, prev[r]), diag);
    if (i == 0 && j == 0) best = 0.f;
    const float v = i < n ? d + best : INFINITY;
    diag = prev[r];                             // D[i][j-1] is the diagonal of the row below
    up = v;
    prev[r] = v;
    row_min = fminf(row_min, v);
    if (i == i_last) cur_r = v;
  }
  return row_min;
}

// D[n-1][m-1] of one pair on one warp: query rows qp[n][dim] (global), template st[m][dim] and the boundary row
// brow[m] in shared memory.  q / q_strip: the caller's registers holding the strip of rows starting at q_strip (a warp
// that keeps one query for many templates loads a one-strip query once).  With PRUNE the pair is abandoned -- the call
// returns false -- as soon as a lower bound on its final cost is strictly greater than `kth`; sufmin[m] is scratch.
template <int R, int DMAX, bool PRUNE>
__device__ __forceinline__ bool dtw_pair(const float* __restrict__ qp, int n, const float* st, int m, int dim, float* brow,
                                         float* sufmin, float kth, float (&q)[R][DMAX], int& q_strip, float& cost) {
  const int lane = threadIdx.x & 31;
  for (int j = lane; j < m; j += 32) brow[j] = INFINITY;      // "row -1"
  __syncwarp();
  float result = INFINITY;
  constexpr int kStrip = 32 * R;
#pragma unroll 1
  for (int i0 = 0; i0 < n; i0 += kStrip) {
    const int ns = min(kStrip, n - i0);         // rows of this strip
    if (q_strip != i0) {                        // this lane's rows of the strip in registers
#pragma unroll
      for (int r = 0; r < R; ++r) {
        const int i = i0 + lane * R + r;
#pragma unroll
        for (int c = 0; c < DMAX; ++c) q[r][c] = (i < n && c < dim) ? qp[(size_t)i * dim + c] : 0.f;
      }
      q_strip = i0;
    }
    if (PRUNE && i0 > 0) {                      // sufmin[j] = min over columns >= j of the previous strip's last row
      float carry = INFINITY;
      for (int base = ((m - 1) >> 5) << 5; base >= 0; base -= 32) {
        const int j = base + lane;
        float v = j < m ? brow[j] : INFINITY;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const float w = __shfl_down_sync(0xffffffffu, v, o); if (lane + o < 32) v = fminf(v, w); }
        v = fminf(v, carry);
        if (j < m) sufmin[j] = v;
        carry = __shfl_sync(0xffffffffu, v, 0);
      }
      __syncwarp();
    }
    const bool final_strip = i0 + ns == n;
    float prev[R];                              // D[i][j-1] of the lane's rows
#pragma unroll
    for (int r = 0; r < R; ++r) prev[r] = INFINITY;
    float top_cur = INFINITY, top_prev = INFINITY;   // D[i-1][j], D[i-1][j-1] from the lane above (lane 0: the boundary row)
    float bottom = INFINITY;                    // D[last row of the lane][j] of the previous step
    float col_min = INFINITY;                   // min of D[i][j] over the strip's rows down to this lane's (PRUNE)
    float last_row_min = INFINITY;              // min over columns <= j of the strip's last row (PRUNE, last lane)
    const int last_lane = (ns - 1) / R;
    const int steps = m + last_lane;
#pragma unroll 1
    for (int s = 0; s < steps; ++s) {
      // the lane above finished column j = s - lane in the previous step
      const float from_above = __shfl_up_sync(0xffffffffu, bottom, 1);
      const float min_above = PRUNE ? __shfl_up_sync(0xffffffffu, col_min, 1) : INFINITY;
      top_prev = top_cur;
      top_cur = lane == 0 ? (s < m ? brow[s] : INFINITY) : from_above;
      const int j = s - lane;
      bool hopeless = false;
      if (j >= 0 && j < m && lane <= last_lane) {
        float cur_r = INFINITY;
        const float row_min = dtw_lane_column<R, DMAX>(q, st + j * dim, dim, i0 + lane * R, n, i0 + ns - 1, j, top_cur, top_prev,
                                                       prev, cur_r);
        bottom = prev[R - 1];
        col_min = lane == 0 ? row_min : fminf(min_above, row_min);
        if (lane == last_lane) {
          brow[j] = cur_r;                      // the strip's last row: top boundary of the next strip
          if (final_strip && j == m - 1) result = cur_r;
          if (PRUNE) {
            // Early exit.  In fp32, v = d + best with d >= 0 rounds to a value >= best, so D never decreases along the
            // predecessor chain of the final cell, and that chain visits every row and every column.  Where it crosses
            // column j it is either (a) in this strip: D >= col_min, the strip's column minimum; (b) above it: it
            // still has to cross the previous strip's last row at a column >= j: D >= sufmin[j]; or (c) below it (not
            // in the final strip): it crossed this strip's last row at a column <= j: D >= last_row_min.  The least
            // of these bounds D[n-1][m-1]; strictly above the k-th cost the pair cannot enter the top k even through
            // the index tie-break.  Under a caller's cost bound U, kth never exceeds ru(U) >= U (rounded up to fp32),
            // so a pair abandoned while the slice's list is short costs more than U and is no candidate either.
            last_row_min = fminf(last_row_min, cur_r);
            float bound = fminf(col_min, i0 > 0 ? sufmin[j] : INFINITY);
            if (!final_strip) bound = fminf(bound, last_row_min);
            hopeless = bound > kth;
          }
        }
      }
      if (PRUNE && __any_sync(0xffffffffu, hopeless)) return false;
    }
    __syncwarp();
  }
  cost = __shfl_sync(0xffffffffu, result, ((n - 1) % kStrip) / R);
  return true;
}

template <int R, int DMAX>
__global__ void __launch_bounds__(32)
dtw_kernel(const float* __restrict__ qf, const int64_t* __restrict__ qoff, int64_t nq, const float* __restrict__ tf,
           const int64_t* __restrict__ toff, int64_t nt, int dim, int max_t_frames, float* __restrict__ cost) {
  extern __shared__ float st[];                 // template frames [m][dim], then the boundary row [max_t_frames]
  float* brow = st + (size_t)max_t_frames * dim;
  const int lane = threadIdx.x;
  const int64_t ti = blockIdx.x, qi = blockIdx.y;
  const int n = (int)(qoff[qi + 1] - qoff[qi]), m = (int)(toff[ti + 1] - toff[ti]);
  float* dst = cost + qi * nt + ti;
  if (n == 0 || m == 0) { if (lane == 0) *dst = INFINITY; return; }
  const float* tp = tf + toff[ti] * dim;
  for (int i = lane; i < m * dim; i += 32) st[i] = tp[i];
  float q[R][DMAX];
  int q_strip = -1;
  float result;
  dtw_pair<R, DMAX, false>(qf + qoff[qi] * dim, n, st, m, dim, brow, nullptr, INFINITY, q, q_strip, result);
  if (lane == 0) *dst = result;
}

// (cost, index) order of every top-k here: ties to the lower template index
__device__ __forceinline__ bool dtw_before(float d, int64_t i, float bd, int64_t bi) { return d < bd || (d == bd && i < bi); }

// The k smallest of `count` candidates (cost, local template index) = get(c) of query qi, on one warp: each lane keeps a
// sorted list of its share, then k rounds of a warp-wide minimum.  Writes (inf, -1, -1) past the valid candidates.
template <class Get>
__device__ __forceinline__ void dtw_warp_select(Get get, int64_t count, int k, int64_t qi, int64_t index_base,
                                                const int32_t* __restrict__ labels, double* __restrict__ nbr_cost,
                                                int64_t* __restrict__ nbr_idx, int32_t* __restrict__ nbr_label) {
  const int lane = threadIdx.x & 31;
  float bd[kKnnMaxK]; int64_t bi[kKnnMaxK];
  for (int c = 0; c < k; ++c) { bd[c] = INFINITY; bi[c] = INT64_MAX; }
  for (int64_t i = lane; i < count; i += 32) {
    float d; int64_t ix;
    get(i, d, ix);
    if (dtw_before(d, ix, bd[k - 1], bi[k - 1])) {
      int s = k - 1;
      while (s > 0 && dtw_before(d, ix, bd[s - 1], bi[s - 1])) { bd[s] = bd[s - 1]; bi[s] = bi[s - 1]; --s; }
      bd[s] = d; bi[s] = ix;
    }
  }
  int head = 0;
  for (int c = 0; c < k; ++c) {
    float md = head < k ? bd[head] : INFINITY;
    int64_t mi = head < k ? bi[head] : INT64_MAX;
    int owner = lane;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float od = __shfl_xor_sync(0xffffffffu, md, o);
      const int64_t oi = __shfl_xor_sync(0xffffffffu, mi, o);
      const int oo = __shfl_xor_sync(0xffffffffu, owner, o);
      if (dtw_before(od, oi, md, mi)) { md = od; mi = oi; owner = oo; }
    }
    if (owner == lane && mi != INT64_MAX) ++head;
    if (lane == 0) {
      const bool valid = mi != INT64_MAX && md < INFINITY;
      if (nbr_cost) nbr_cost[qi * k + c] = valid ? (double)md : INFINITY;
      if (nbr_idx) nbr_idx[qi * k + c] = valid ? index_base + mi : -1;
      if (nbr_label) nbr_label[qi * k + c] = valid ? labels[mi] : -1;
    }
  }
}

// k smallest costs per query (ties to the lower template index): one warp per query
__global__ void dtw_topk_kernel(const float* __restrict__ cost, int64_t nq, int64_t nt, int k, int64_t index_base,
                                const int32_t* __restrict__ labels, double* __restrict__ nbr_cost,
                                int64_t* __restrict__ nbr_idx, int32_t* __restrict__ nbr_label) {
  const int64_t qi = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (qi >= nq) return;
  const float* row = cost + qi * nt;
  dtw_warp_select([&](int64_t i, float& d, int64_t& ix) { d = row[i]; ix = i; }, nt, k, qi, index_base, labels, nbr_cost,
                  nbr_idx, nbr_label);
}

// DTW with the top-k fused in and no cost matrix: one warp per (query, slice of templates).  The warp scores its slice's
// templates one after another (dtw_pair with PRUNE) and keeps the slice's k best (cost, index) pairs in registers, entry
// c on lane c, so the k-th cost that decides the early exit is one shuffle away.  Output: cand_d / cand_i [unit][k],
// (inf, INT64_MAX) where the slice has fewer than k, merged per query by dtw_merge_kernel.  stats[0] / [1] count the
// pairs scored to the last cell / abandoned.
// bound (nullable, float64 per query): only templates with cost <= bound[qi] (compared in float64) are candidates, and
// the abandon threshold starts at the bound rounded up to fp32 instead of inf.  A bound that is not >= 0 (negative,
// NaN) admits nothing: the slice is skipped and its pairs count as abandoned.  +inf (or no array) is no bound.
template <int R, int DMAX>
__global__ void __launch_bounds__(kDtwFusedWarps * 32, 1)
dtw_topk_fused_kernel(const float* __restrict__ qf, const int64_t* __restrict__ qoff, const int32_t* __restrict__ qlen, int64_t nq,
                      const float* __restrict__ tf, const int64_t* __restrict__ toff, const int32_t* __restrict__ tlen,
                      int64_t nt, int dim, int max_t_frames, int slices, int k, const double* __restrict__ bound,
                      float* __restrict__ cand_d, int64_t* __restrict__ cand_i, unsigned long long* __restrict__ stats) {
  extern __shared__ float smem[];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int64_t unit = (int64_t)blockIdx.x * (blockDim.x >> 5) + w;
  if (unit >= nq * slices) return;              // whole warps only: no CTA-wide barrier below
  const int64_t qi = unit / slices, sl = unit % slices;
  float* st = smem + (size_t)w * ((size_t)max_t_frames * (dim + 2));   // template [m][dim], boundary row, suffix minima
  float* brow = st + (size_t)max_t_frames * dim;
  float* sufmin = brow + max_t_frames;
  const int n = qlen ? qlen[qi] : (int)(qoff[qi + 1] - qoff[qi]);
  const float* qp = qf + qoff[qi] * dim;
  const int64_t t_end = nt * (sl + 1) / slices;
  const double ub = bound ? bound[qi] : (double)INFINITY;
  const float kth0 = __double2float_ru(ub);     // ub <= kth0: a lower bound above kth0 puts the cost above ub
  float my_d = INFINITY, kth = kth0;
  int64_t my_i = INT64_MAX;
  float q[R][DMAX];
  int q_strip = -1;
  unsigned long long scored = 0, abandoned = 0;
  int64_t ti = nt * sl / slices;
  if (!(ub >= 0)) { abandoned = t_end - ti; ti = t_end; }
#pragma unroll 1
  for (; ti < t_end; ++ti) {
    const int m = tlen[ti];
    float cost = INFINITY;
    if (n > 0 && m > 0) {
      const float* tp = tf + toff[ti] * dim;
      __syncwarp();                             // the previous pair is done with st
      for (int i = lane; i < m * dim; i += 32) st[i] = tp[i];
      if (!dtw_pair<R, DMAX, true>(qp, n, st, m, dim, brow, sufmin, kth, q, q_strip, cost)) { ++abandoned; continue; }
    }
    ++scored;
    // insert into the sorted list held one entry per lane; the bound is compared in float64, since kth0 may admit
    // costs in (ub, kth0]
    if (cost <= kth && (double)cost <= ub) {
      const bool before = dtw_before(cost, ti, my_d, my_i);
      const bool shift = __shfl_up_sync(0xffffffffu, (int)before, 1) && lane > 0;
      const float up_d = __shfl_up_sync(0xffffffffu, my_d, 1);
      const int64_t up_i = __shfl_up_sync(0xffffffffu, my_i, 1);
      if (lane < k) {
        if (shift) { my_d = up_d; my_i = up_i; }
        else if (before) { my_d = cost; my_i = ti; }
      }
      kth = fminf(kth0, __shfl_sync(0xffffffffu, my_d, k - 1));   // a short list must not lift it to inf
    }
  }
  if (lane < k) { cand_d[unit * k + lane] = my_d; cand_i[unit * k + lane] = my_i; }
  if (lane == 0) { atomicAdd(stats, scored); atomicAdd(stats + 1, abandoned); }
}

// the slices' candidates of one query -> its top k: one warp per query, dtw_topk_kernel's selection
__global__ void dtw_merge_kernel(const float* __restrict__ cand_d, const int64_t* __restrict__ cand_i, int64_t nq, int slices,
                                 int k, int64_t index_base, const int32_t* __restrict__ labels, double* __restrict__ nbr_cost,
                                 int64_t* __restrict__ nbr_idx, int32_t* __restrict__ nbr_label) {
  const int64_t qi = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (qi >= nq) return;
  const int64_t base = qi * slices * k;
  dtw_warp_select([&](int64_t i, float& d, int64_t& ix) { d = cand_d[base + i]; ix = cand_i[base + i]; }, (int64_t)slices * k, k,
                  qi, index_base, labels, nbr_cost, nbr_idx, nbr_label);
}

}  // namespace

size_t mfcc_smem_bytes(int n_fft, int n_mels) { return (size_t)n_fft * 8 + (size_t)(n_fft / 2 + 1) * 4 + (size_t)n_mels * 4 + 16; }

cudaError_t launch_mfcc(const int16_t* samples, const int64_t* offsets, const int32_t* lengths, const int32_t* seg_start,
                        const int32_t* seg_end, int64_t n_utts, const MfccArgs& a, const float* window, const float2* twiddle,
                        const float* filterbank, const int2* fb_range, const float* dct, const int64_t* mfcc_offsets, float* out,
                        int32_t* n_frames_out, unsigned int* work_counter, int sm_count, cudaStream_t st) {
  if (n_utts == 0) return cudaSuccess;
  const size_t smem = mfcc_smem_bytes(a.n_fft, a.n_mels);
  cudaError_t e = cudaFuncSetAttribute(mfcc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  cudaMemsetAsync(work_counter, 0, sizeof(unsigned int), st);
  const int grid = (int)std::min<int64_t>(n_utts, (int64_t)sm_count * 4);
  mfcc_kernel<<<grid, kMfccThreads, smem, st>>>(samples, offsets, lengths, seg_start, seg_end, n_utts, a, window, twiddle,
                                                filterbank, fb_range, dct, mfcc_offsets, out, n_frames_out, work_counter);
  return cudaGetLastError();
}

int dtw_max_query_frames() { return INT32_MAX; }      // any length: strips of 32 R rows
int dtw_max_dim() { return kDtwMaxDim; }
size_t dtw_smem_bytes(int max_t_frames, int dim) { return ((size_t)std::max(max_t_frames, 1) * dim + (size_t)std::max(max_t_frames, 1)) * sizeof(float); }

namespace {
// The (R, DMAX) build for a feature dimension and a query length: DMAX the smallest register row that holds a frame,
// R the largest strip the registers allow (R * DMAX <= 128), and for the 13 MFCCs the smallest strip that holds the
// longest query -- a strip with idle lanes costs R per step where one of 32 R rows costs 1.  Any build gives the same
// bits: padded features add fmaf(0, 0, d2) = d2, and strips only change where a row is held.
template <class F>
cudaError_t dtw_build(int dim, int max_q_frames, F&& f) {
  using std::integral_constant;
  if (dim > 64) return f(integral_constant<int, 1>{}, integral_constant<int, 128>{});
  if (dim > 32) return f(integral_constant<int, 2>{}, integral_constant<int, 64>{});
  if (dim > 16) return f(integral_constant<int, 4>{}, integral_constant<int, 32>{});
  if (max_q_frames <= 32) return f(integral_constant<int, 1>{}, integral_constant<int, 16>{});
  if (max_q_frames <= 64) return f(integral_constant<int, 2>{}, integral_constant<int, 16>{});
  if (max_q_frames <= 128) return f(integral_constant<int, 4>{}, integral_constant<int, 16>{});
  return f(integral_constant<int, 8>{}, integral_constant<int, 16>{});
}
}  // namespace

cudaError_t launch_dtw(const float* qf, const int64_t* qoff, int64_t nq, int max_q_frames, const float* tf, const int64_t* toff,
                       int64_t nt, int max_t_frames, int dim, float* cost, cudaStream_t st) {
  if (nq == 0 || nt == 0) return cudaSuccess;
  if (dim > kDtwMaxDim) return cudaErrorInvalidValue;
  const size_t smem = dtw_smem_bytes(max_t_frames, dim);
  // grid.y is limited to 65535: queries are processed in slabs
  for (int64_t q0 = 0; q0 < nq; q0 += 65535) {
    const int64_t qc = std::min<int64_t>(65535, nq - q0);
    const dim3 grid((unsigned)nt, (unsigned)qc);
    const float* cq = qf; const int64_t* oq = qoff + q0; float* cc = cost + q0 * nt;
    cudaError_t e = dtw_build(dim, max_q_frames, [&](auto r, auto d) -> cudaError_t {
      auto kern = dtw_kernel<decltype(r)::value, decltype(d)::value>;
      cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) return e;
      kern<<<grid, 32, smem, st>>>(cq, oq, qc, tf, toff, nt, dim, std::max(max_t_frames, 1), cc);
      return cudaGetLastError();
    });
    if (e != cudaSuccess) return e;
  }
  return cudaSuccess;
}

size_t dtw_fused_smem_per_warp(int max_t_frames, int dim) { return (size_t)std::max(max_t_frames, 1) * (dim + 2) * sizeof(float); }
int dtw_fused_max_warps() { return kDtwFusedWarps; }

int64_t dtw_fused_units(int64_t nq, int sm_count) { return std::max<int64_t>(nq, (int64_t)sm_count * 32); }

int dtw_fused_slices(int64_t nq, int64_t nt, int sm_count) {
  // enough (query, slice) warps for a few waves when queries are few, but slices of >= 32 templates so that the k-th
  // cost is known early; nq * slices <= dtw_fused_units(nq): scratch sized for nq serves every smaller call
  if (nq < 1) return 1;
  const int64_t by_units = dtw_fused_units(nq, sm_count) / nq;
  return (int)std::max<int64_t>(1, std::min<int64_t>(by_units, nt / 32));
}

cudaError_t launch_dtw_topk_fused(const float* qf, const int64_t* qoff, const int32_t* qlen, int64_t nq, int max_q_frames,
                                  const float* tf, const int64_t* toff, const int32_t* tlen, int64_t nt, int max_t_frames, int dim,
                                  int k, const double* bound, int slices, int warps, int64_t index_base, const int32_t* labels,
                                  float* cand_d, int64_t* cand_i, unsigned long long* stats, double* nbr_cost,
                                  int64_t* nbr_idx, int32_t* nbr_label, cudaStream_t st) {
  cudaError_t e = cudaMemsetAsync(stats, 0, 2 * sizeof(unsigned long long), st);
  if (e != cudaSuccess || nq == 0) return e;
  if (dim > kDtwMaxDim || k < 1 || k > kKnnMaxK || warps < 1 || warps > kDtwFusedWarps) return cudaErrorInvalidValue;
  const int mt = std::max(max_t_frames, 1);
  const size_t smem = dtw_fused_smem_per_warp(mt, dim) * warps;
  const int64_t units = nq * slices;
  e = dtw_build(dim, max_q_frames > 0 ? max_q_frames : 128, [&](auto r, auto d) -> cudaError_t {
    auto kern = dtw_topk_fused_kernel<decltype(r)::value, decltype(d)::value>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kern<<<(unsigned)((units + warps - 1) / warps), 32 * warps, smem, st>>>(qf, qoff, qlen, nq, tf, toff, tlen, nt, dim, mt,
                                                                            slices, k, bound, cand_d, cand_i, stats);
    return cudaGetLastError();
  });
  if (e != cudaSuccess) return e;
  dtw_merge_kernel<<<(unsigned)((nq + 7) / 8), 256, 0, st>>>(cand_d, cand_i, nq, slices, k, index_base, labels, nbr_cost, nbr_idx,
                                                            nbr_label);
  return cudaGetLastError();
}

cudaError_t launch_dtw_topk(const float* cost, int64_t nq, int64_t nt, int k, int64_t index_base, const int32_t* labels,
                            double* nbr_cost, int64_t* nbr_idx, int32_t* nbr_label, cudaStream_t st) {
  if (nq == 0) return cudaSuccess;
  dtw_topk_kernel<<<(unsigned)((nq + 7) / 8), 256, 0, st>>>(cost, nq, nt, k, index_base, labels, nbr_cost, nbr_idx, nbr_label);
  return cudaGetLastError();
}

}  // namespace dsp
