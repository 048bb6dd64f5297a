// Shared device helpers for libdspfront (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/dspfront.h"

namespace dsp {

constexpr int kStats = 15;

// ---------------------------------------------------------------------------
// NumPy's pairwise summation, restated so that float64 sums are bit-identical
// to np.sum / np.mean on a contiguous 1-D array (numpy/_core/src/umath/
// loops_utils.h.src, @TYPE@_pairwise_sum): < 8 terms sequential; <= 128 terms
// eight interleaved accumulators combined as ((0+1)+(2+3))+((4+5)+(6+7)) then the
// tail; otherwise split at n/2 rounded down to a multiple of 8.  `term(i)` yields
// the i-th addend.  Used wherever a sum feeds an integer decision of the
// reference (endpoint thresholds, audio_processing.py:186-217).
// ---------------------------------------------------------------------------
template <class Term>
__device__ __forceinline__ double np_pairwise_leaf(Term term, int64_t off, int n) {
  if (n < 8) {
    double r = 0.0;
    for (int i = 0; i < n; ++i) r += term(off + i);
    return r;
  }
  double r0 = term(off + 0), r1 = term(off + 1), r2 = term(off + 2), r3 = term(off + 3);
  double r4 = term(off + 4), r5 = term(off + 5), r6 = term(off + 6), r7 = term(off + 7);
  int i = 8;
  const int body = n - (n % 8);
  for (; i < body; i += 8) {
    r0 += term(off + i + 0); r1 += term(off + i + 1); r2 += term(off + i + 2); r3 += term(off + i + 3);
    r4 += term(off + i + 4); r5 += term(off + i + 5); r6 += term(off + i + 6); r7 += term(off + i + 7);
  }
  double res = ((r0 + r1) + (r2 + r3)) + ((r4 + r5) + (r6 + r7));
  for (; i < n; ++i) res += term(off + i);
  return res;
}

constexpr int kPairwiseBlock = 128;
constexpr int kPairwiseDepth = 40;

template <class Term>
__device__ double np_pairwise_sum(Term term, int64_t n) {
  if (n <= kPairwiseBlock) return np_pairwise_leaf(term, 0, (int)n);
  int64_t st_off[kPairwiseDepth];
  int64_t st_n[kPairwiseDepth];
  double st_left[kPairwiseDepth];
  int8_t st_state[kPairwiseDepth];
  int sp = 0;
  st_off[0] = 0; st_n[0] = n; st_state[0] = 0;
  double ret = 0.0;
  bool have = false;
  while (sp >= 0) {
    if (have) {
      if (st_state[sp] == 1) {            // left child finished: descend into the right one
        st_left[sp] = ret;
        st_state[sp] = 2;
        have = false;
        int64_t n2 = st_n[sp] / 2; n2 -= n2 % 8;
        st_off[sp + 1] = st_off[sp] + n2; st_n[sp + 1] = st_n[sp] - n2; st_state[sp + 1] = 0;
        ++sp;
      } else {                            // right child finished
        ret = st_left[sp] + ret;
        --sp;
      }
    } else {
      const int64_t nn = st_n[sp];
      if (nn <= kPairwiseBlock) {
        ret = np_pairwise_leaf(term, st_off[sp], (int)nn);
        have = true;
        --sp;
      } else {
        st_state[sp] = 1;
        int64_t n2 = nn / 2; n2 -= n2 % 8;
        st_off[sp + 1] = st_off[sp]; st_n[sp + 1] = n2; st_state[sp + 1] = 0;
        ++sp;
      }
    }
  }
  return ret;
}

// np.mean of the <= 10 noise frames of endpoint detection in NumPy's association (audio_processing.py:188-195;
// pairwise: < 8 terms sequential, else eight accumulators combined as a tree, then the tail) -- out of line, it is
// cold code.
static __device__ __noinline__ double noise_mean(const double* v, int n) {
  double r;
  if (n < 8) { r = 0.0; for (int i = 0; i < n; ++i) r += v[i]; }
  else { r = ((v[0] + v[1]) + (v[2] + v[3])) + ((v[4] + v[5]) + (v[6] + v[7])); for (int i = 8; i < n; ++i) r += v[i]; }
  return r / (double)n;
}

// the low 16-bit half of a word of two int16 PCM samples, sign-extended (the high half is (int)w >> 16)
__device__ __forceinline__ int sext16(uint32_t w) { return (int)(short)(w & 0xffffu); }

// np.percentile(..., method='linear') interpolation between the two order statistics
// (numpy/lib/_function_base_impl.py:4671-4675): a + (b-a)*g, or b - (b-a)*(1-g) when g >= 0.5.
__device__ __forceinline__ double np_lerp(double a, double b, double g) {
  const double d = b - a;
  return (g >= 0.5) ? (b - d * (1.0 - g)) : (a + d * g);
}

// Order-preserving map double -> uint64 (handles negatives; NaNs sort last).
__device__ __forceinline__ uint64_t f64_key(double v) {
  uint64_t u = (uint64_t)__double_as_longlong(v);
  return (u & 0x8000000000000000ull) ? ~u : (u | 0x8000000000000000ull);
}
__device__ __forceinline__ double key_f64(uint64_t k) {
  uint64_t u = (k & 0x8000000000000000ull) ? (k & 0x7fffffffffffffffull) : ~k;
  return __longlong_as_double((long long)u);
}

// ---------------------------------------------------------------------------
// Block-wide helpers (any power-of-two-free block size that is a multiple of 32).
// `sh` must hold at least 64 doubles / 64 uint64.
// ---------------------------------------------------------------------------
__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }
__device__ __forceinline__ int warp_id() { return threadIdx.x >> 5; }

template <class T, class Op>
__device__ __forceinline__ T warp_reduce(T v, Op op) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    T other = __shfl_xor_sync(0xffffffffu, v, o);
    v = op(v, other);
  }
  return v;
}

// All threads must call; result valid in every thread.
template <class T, class Op>
__device__ T block_reduce(T v, Op op, T identity, T* sh) {
  v = warp_reduce(v, op);
  __syncthreads();
  if (lane_id() == 0) sh[warp_id()] = v;
  __syncthreads();
  const int nw = (blockDim.x + 31) >> 5;
  T r = (threadIdx.x < nw) ? sh[threadIdx.x] : identity;
  if (warp_id() == 0) {
    r = warp_reduce(r, op);
    if (lane_id() == 0) sh[0] = r;
  }
  __syncthreads();
  r = sh[0];
  __syncthreads();
  return r;
}

struct OpAddD { __device__ double operator()(double a, double b) const { return a + b; } };
struct OpMaxD { __device__ double operator()(double a, double b) const { return a > b ? a : b; } };
struct OpMinD { __device__ double operator()(double a, double b) const { return a < b ? a : b; } };
struct OpAddLL { __device__ long long operator()(long long a, long long b) const { return a + b; } };
struct OpMaxI { __device__ int operator()(int a, int b) const { return a > b ? a : b; } };
struct OpMinI { __device__ int operator()(int a, int b) const { return a < b ? a : b; } };
struct OpMinU64 { __device__ unsigned long long operator()(unsigned long long a, unsigned long long b) const { return a < b ? a : b; } };
struct OpAddI { __device__ int operator()(int a, int b) const { return a + b; } };

// ---------------------------------------------------------------------------
// Block-wide order statistics by MSD radix select on 64-bit keys.
// get(i) returns the i-th key (i < n).  Returns the keys of rank r and r+1
// (0-based, ascending; rank r+1 clamps to r when r == n-1).  hist: 256 ints of
// shared memory, sh: 64 uint64 of shared memory.  All threads must call.
// ---------------------------------------------------------------------------
template <class Get>
__device__ void block_select_pair(Get get, int n, int r, int* hist, unsigned long long* sh,
                                  uint64_t* k_lo, uint64_t* k_hi) {
  uint64_t prefix = 0, mask = 0;
  int rank = r;
  __shared__ int s_digit, s_rank;
  for (int shift = 56; shift >= 0; shift -= 8) {
    for (int i = threadIdx.x; i < 256; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      const uint64_t k = get(i);
      if ((k & mask) == prefix) atomicAdd(&hist[(int)((k >> shift) & 0xff)], 1);
    }
    __syncthreads();
    if (threadIdx.x < 32) {
      int c[8], tot = 0;
#pragma unroll
      for (int j = 0; j < 8; ++j) { c[j] = hist[threadIdx.x * 8 + j]; tot += c[j]; }
      int incl = tot;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        int t = __shfl_up_sync(0xffffffffu, incl, o);
        if ((int)threadIdx.x >= o) incl += t;
      }
      int run = incl - tot;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        if (rank >= run && rank < run + c[j]) { s_digit = threadIdx.x * 8 + j; s_rank = rank - run; }
        run += c[j];
      }
    }
    __syncthreads();
    prefix |= ((uint64_t)s_digit) << shift;
    mask |= 0xffull << shift;
    rank = s_rank;
    __syncthreads();
  }
  const uint64_t sel = prefix;
  // rank r+1: equal to sel when more than (r+1) keys are <= sel, else the smallest key above it.
  int le = 0;
  unsigned long long nxt = ~0ull;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const uint64_t k = get(i);
    if (k <= sel) ++le; else if (k < nxt) nxt = k;
  }
  le = block_reduce<int>(le, OpAddI(), 0, reinterpret_cast<int*>(sh));
  nxt = block_reduce<unsigned long long>(nxt, OpMinU64(), ~0ull, sh);
  *k_lo = sel;
  *k_hi = (le >= r + 2 || nxt == ~0ull) ? sel : (uint64_t)nxt;
}

}  // namespace dsp
