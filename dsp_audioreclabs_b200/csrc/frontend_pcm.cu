// Fused front-end kernel for 16-bit mono PCM (the throughput path).
//
// One CTA owns one utterance at a time (persistent grid, dynamic work counter).  The
// utterance is brought into shared memory ONCE with 1-D bulk async copies (TMA,
// cp.async.bulk + mbarrier) and every later stage reads shared memory only, so frame
// overlap and the reference's two framing passes cost no extra HBM traffic:
//
//   P1  sum / min / max of the PCM codes            -> DC (exact rational S/N), peak
//   P2  per 64-sample group: sum d, sum d^2 (exact integers, d = k - thr with
//       thr = floor(S/N)+1, so "sample above the mean" is just d >= 0) and one sign bit per
//       sample                                       -> every EPD frame from group sums
//   P3  endpoint decision: 90th percentile by a warp-level radix select, thresholds, six
//       ballot-style searches; a certified-margin test flags utterances for the float64 replay
//   P4  windowed energy / magnitude over the trimmed frames (fp32 FMA); for hop 128 / length
//       256 a sample-stationary chain (each sample converted once, window in registers),
//       otherwise 8 lanes per frame; zero-crossing counts by popcount over the sign bits
//   P5  mean / std / max / min / median of the three sequences, one warp per sequence
//
// Exactness (DESIGN.md "numerics"): with PCM input the reference's float64 values are
// x_i = k_i/32768, so sign(x_i - mean) == sign(N*k_i - S) and sum((x_i-mean)/peak)^2 over a
// frame equals (sum d^2 - 2*phi*sum d + fl*phi^2) * (N/M)^2 with integers N, S, M and
// phi = S/N - thr in [-1, 0): zero-crossing counts are exact and EPD energies are within a few
// ulp of the real-number value.  Threshold comparisons closer than a rigorous bound on the
// reference's own rounding are not decided here but replayed in float64 NumPy order.
//
// Reference: src/audio_processing.py:49-90,135-275,299-333; src/feature_extraction.py:12-88.
#include "kernels.cuh"
#include "ptx.cuh"

namespace dsp {

namespace {

constexpr int kGroup = 64;          // samples per group-sum record
constexpr int kLanesPerFrame = 8;   // generic P4: lanes cooperating on one frame

struct SmemLayout {
  int samples, bits, g2, g1, e, z, win, hist, cand, sh, misc, total;
};

__host__ __device__ inline int align16(int x) { return (x + 15) & ~15; }

__host__ __device__ inline SmemLayout make_layout(int cap_samples, int cap_frames, int fl, bool resident) {
  SmemLayout L;
  const int ng = cap_samples / kGroup;
  int o = 0;
  L.samples = o; o += resident ? align16(2 * cap_samples + 32) : 0;
  L.bits = o;    o += align16(4 * (cap_samples / 32 + 4));
  // group sums; the same region later holds the three float feature sequences
  const int gbytes = 12 * ng, fbytes = 12 * cap_frames;
  L.g2 = o;
  L.g1 = o + 8 * ng;
  o += align16(gbytes > fbytes ? gbytes : fbytes);
  L.e = o;       o += align16(8 * cap_frames);
  L.z = o;       o += align16(4 * cap_frames);
  L.win = o;     o += align16(4 * fl);
  L.hist = o;    o += 3 * 256 * 4;
  L.cand = o;    o += 3 * 64 * 4;
  L.sh = o;      o += 64 * 8;
  L.misc = o;    o += 384;
  L.total = o;
  return L;
}

// ---- sign-bit string helpers ----------------------------------------------------------
__device__ __forceinline__ int bit_at(const uint32_t* bits, int i) { return (bits[i >> 5] >> (i & 31)) & 1; }

// number of i in [p, q-1) with bit[i] != bit[i+1]  (sign changes among samples p..q-1)
__device__ __forceinline__ int count_changes(const uint32_t* bits, int p, int q) {
  if (q - p < 2) return 0;
  int c = 0;
  if (((p | q) & 31) == 0) {               // word-aligned frame: no edge masks except the last pair
    const int w0 = p >> 5, w1 = (q >> 5) - 1;
    uint32_t cur = bits[w0];
    for (int w = w0; w < w1; ++w) {
      const uint32_t nxt = bits[w + 1];
      c += __popc(cur ^ __funnelshift_r(cur, nxt, 1));
      cur = nxt;
    }
    c += __popc((cur ^ (cur >> 1)) & 0x7fffffffu);
    return c;
  }
  const int last = q - 2;  // last pair start
  const int w0 = p >> 5, w1 = last >> 5;
  #pragma unroll 1
  for (int w = w0; w <= w1; ++w) {
    const uint32_t cur = bits[w], nxt = bits[w + 1];
    uint32_t x = cur ^ __funnelshift_r(cur, nxt, 1);
    if (w == w0) x &= 0xffffffffu << (p & 31);
    if (w == w1) x &= 0xffffffffu >> (31 - (last & 31));
    c += __popc(x);
  }
  return c;
}

// zero crossings of one windowed frame (compute_zero_crossing_rate on frame*window,
// audio_processing.py:119-132): zero-padded samples and Hanning's exact-zero end points count
// as negative.
__device__ __noinline__ int frame_zcr(const uint32_t* bits, int p, int valid, int fl, bool hann) {
  if (hann && fl <= 2) return 0;
  int zc = count_changes(bits, p, p + valid);
  if (valid < fl) zc += bit_at(bits, p + valid - 1);
  if (hann) {
    const int s0 = bit_at(bits, p), s1 = valid > 1 ? bit_at(bits, p + 1) : 0;
    zc += s1 - (s0 ^ s1);
    if (fl - 1 < valid) {
      const int sl = bit_at(bits, p + fl - 1), sp = bit_at(bits, p + fl - 2);
      zc += sp - (sp ^ sl);
    }
  }
  return zc;
}

struct UttConst {
  int thr;         // floor(S/N) + 1: sample is above the mean iff k >= thr
  float phi;       // S/N - thr, in [-1, 0)
  double phi_d;
  double inv_m;    // N/M (1 when the signal is constant)
  double mu;       // S/N
};

// ---- named barriers (warp-specialised roles) --------------------------------------------
constexpr int kBarMain = 1;       // main warps only
constexpr int kBarFeatFull = 2;   // main arrive, stats wait: feature sequences are in shared memory
constexpr int kBarFeatEmpty = 3;  // stats arrive, main wait: feature sequences have been consumed
constexpr int kStatsRegs = 11;    // feature frames per lane held in registers by the stats warps

// Radix-select bookkeeping shared by the block- and warp-level selects: after the 256-bin
// histogram of (key - lo) >> s is in `hist`, one warp finds the bin holding `rank`.
__device__ __forceinline__ void scan_bins(const int* hist, int lane, int rank, int* digit_out, int* rank_out, int* cnt_out) {
  int c[8], tot = 0;
#pragma unroll
  for (int j = 0; j < 8; ++j) { c[j] = hist[lane * 8 + j]; tot += c[j]; }
  int incl = tot;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
  int run = incl - tot, digit = -1, newrank = 0, newcnt = 0;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    if (digit < 0 && rank >= run && rank < run + c[j]) { digit = lane * 8 + j; newrank = rank - run; newcnt = c[j]; }
    run += c[j];
  }
  const int src = __ffs(__ballot_sync(0xffffffffu, digit >= 0)) - 1;
  *digit_out = __shfl_sync(0xffffffffu, digit, src);
  *rank_out = __shfl_sync(0xffffffffu, newrank, src);
  *cnt_out = __shfl_sync(0xffffffffu, newcnt, src);
}

__device__ __forceinline__ int first_shift(uint32_t kmin, uint32_t kmax) {
  const uint32_t span = kmax - kmin;
  const int bits = 32 - __clz(span);          // 0 when all keys are equal
  return bits > 8 ? bits - 8 : 0;
}

// ---------------------------------------------------------------------------------------
// Statistics of one non-negative float sequence by ONE warp (compute_statistics,
// feature_extraction.py:46-62): mean, population std, max, min and the median by a radix select
// whose first pass spreads 256 bins over [min, max] of the float bit patterns.  vals[j * stride]
// is element lane + 32*j of the sequence (a per-lane array in local memory, or the sequence itself
// in shared memory).  Deliberately NOT inlined: it runs on the statistics warps only, once per
// sequence, and three unrolled copies of it used to blow the instruction cache for the main warps.
// ---------------------------------------------------------------------------------------
__device__ __noinline__ void warp_sequence_stats(const float* vals, int stride, int n, int* hist, float* cand, float* out5) {
  const int lane = threadIdx.x & 31;
  const int nj = (n + 31) / 32;
  double sum = 0.0;
  float mx = 0.f, mn = INFINITY;
#pragma unroll 1
  for (int j = 0; j < nj; ++j) if (lane + 32 * j < n) { const float x = vals[j * stride]; sum += (double)x; mx = fmaxf(mx, x); mn = fminf(mn, x); }
  sum = warp_reduce(sum, OpAddD());
  mx = warp_reduce(mx, [](float x, float y) { return fmaxf(x, y); });
  mn = warp_reduce(mn, [](float x, float y) { return fminf(x, y); });
  const double mean = sum / (double)n;
  double ss = 0.0;
#pragma unroll 1
  for (int j = 0; j < nj; ++j) if (lane + 32 * j < n) { const double d = (double)vals[j * stride] - mean; ss += d * d; }
  ss = warp_reduce(ss, OpAddD());

  uint32_t lo = __float_as_uint(mn);
  int s = first_shift(lo, __float_as_uint(mx));
  int s_used = 32, rank = (n - 1) / 2, cnt = n;
  while (cnt > 32) {
#pragma unroll 1
    for (int j = 0; j < 8; ++j) hist[lane * 8 + j] = 0;
    __syncwarp();
#pragma unroll 1
    for (int j = 0; j < nj; ++j) if (lane + 32 * j < n) {
      const uint32_t k = __float_as_uint(vals[j * stride]);
      if (k >= lo) { const uint32_t d = (k - lo) >> s; if (d < 256u) atomicAdd(&hist[d], 1); }
    }
    __syncwarp();
    int digit;
    scan_bins(hist, lane, rank, &digit, &rank, &cnt);
    lo += (uint32_t)digit << s;
    s_used = s;
    __syncwarp();
    if (s == 0) break;
    s = s > 8 ? s - 8 : 0;
  }
  const unsigned long long span = 1ull << s_used;
  float sel, sel2;
  bool have2;
  if (cnt > 32) {                     // s == 0: every candidate has the same bit pattern
    sel = sel2 = __uint_as_float(lo);
    have2 = rank + 1 < cnt;
  } else {
    if (lane == 0) hist[0] = 0;
    __syncwarp();
#pragma unroll 1
    for (int j = 0; j < nj; ++j) if (lane + 32 * j < n) {
      const float x = vals[j * stride];
      const uint32_t k = __float_as_uint(x);
      if (n <= 32 || (k >= lo && (unsigned long long)(k - lo) < span)) cand[atomicAdd(&hist[0], 1)] = x;
    }
    __syncwarp();
    const float mine = lane < cnt ? cand[lane] : INFINITY;
    int below = 0;
#pragma unroll 1
    for (int j = 0; j < cnt; ++j) {
      const float o = __shfl_sync(0xffffffffu, mine, j);
      below += (o < mine) || (o == mine && j < lane);
    }
    const unsigned m1 = __ballot_sync(0xffffffffu, lane < cnt && below == rank);
    const unsigned m2 = __ballot_sync(0xffffffffu, lane < cnt && below == rank + 1);
    sel = __shfl_sync(0xffffffffu, mine, __ffs(m1) - 1);
    have2 = m2 != 0;
    sel2 = have2 ? __shfl_sync(0xffffffffu, mine, __ffs(m2) - 1) : sel;
    __syncwarp();
  }
  if (!have2 && !(n & 1)) {           // upper middle lies above the candidate bin
    float nxt = INFINITY;
#pragma unroll 1
    for (int j = 0; j < nj; ++j) if (lane + 32 * j < n) { const float x = vals[j * stride]; if (x > sel) nxt = fminf(nxt, x); }
    nxt = warp_reduce(nxt, [](float x, float y) { return fminf(x, y); });
    sel2 = nxt == INFINITY ? sel : nxt;
  }
  if (lane == 0) {
    out5[0] = (float)mean;
    out5[1] = (float)sqrt(ss / (double)n);
    out5[2] = mx; out5[3] = mn;
    out5[4] = (n & 1) ? sel : (float)(((double)sel + (double)sel2) * 0.5);
  }
}

}  // namespace

size_t pcm_kernel_smem_bytes(int cap_samples, int cap_frames, int fl, bool resident) {
  return (size_t)make_layout(cap_samples, cap_frames, fl, resident).total;
}

// kStream: samples are read straight from global memory (pass P1 from HBM, the later passes hit
// L2) instead of being staged in shared memory: ~20 KB of shared memory per CTA instead of
// ~112 KB, so more independent utterance pipelines fit on an SM.  Requires 16-byte aligned
// utterance starts (layout_hint); anything else is replayed by the float64 kernel.
template <bool kStream, int kThreads, int kStatsWarps, int kMinBlocks>
__global__ void __launch_bounds__(kThreads, kMinBlocks)
frontend_pcm_kernel(const PcmArgs a) {
  constexpr int kWarps = kThreads / 32;
  constexpr int kMainWarps = kWarps - kStatsWarps;
  constexpr int kMainThreads = kMainWarps * 32;
  auto main_sync = [&]() { bar_sync(kBarMain, kMainThreads); };
  // Serial sections run on the LAST main warp: the warp scheduler favours higher warp ids, and a lone
  // low-id warp is starved by the other CTA's busy warps (measured: 7.8k cycles for ~300 instructions)
  constexpr int kLeadWarp = kMainWarps - 1;
  constexpr int kLeadTid = kLeadWarp * 32;
  extern __shared__ __align__(128) unsigned char smem[];
  const SmemLayout L = make_layout(a.cap_samples, a.cap_frames, a.fl, !kStream);
  int16_t* s_x = reinterpret_cast<int16_t*>(smem + L.samples);
  uint32_t* s_bits = reinterpret_cast<uint32_t*>(smem + L.bits);
  unsigned long long* s_g2 = reinterpret_cast<unsigned long long*>(smem + L.g2);
  int* s_g1 = reinterpret_cast<int*>(smem + L.g1);
  float* s_fe = reinterpret_cast<float*>(smem + L.g2);            // aliases the group sums
  float* s_fm = s_fe + a.cap_frames;
  float* s_fz = s_fm + a.cap_frames;
  double* s_e = reinterpret_cast<double*>(smem + L.e);
  int* s_z = reinterpret_cast<int*>(smem + L.z);
  float* s_win = reinterpret_cast<float*>(smem + L.win);
  int* s_hist = reinterpret_cast<int*>(smem + L.hist);            // [0] main, [1],[2] stats warps
  float* s_cand = reinterpret_cast<float*>(smem + L.cand);        // 3 x 64 floats
  unsigned long long* s_sh = reinterpret_cast<unsigned long long*>(smem + L.sh);
  // misc block: [0] mbarrier, scalars, mailbox main -> stats
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(smem + L.misc);
  int* s_int = reinterpret_cast<int*>(smem + L.misc + 16);         // 24 ints
  double* s_dbl = reinterpret_cast<double*>(smem + L.misc + 128);  // 16 doubles
  int* s_mail = reinterpret_cast<int*>(smem + L.misc + 256);       // 2 x 8 ints

  const int tid = threadIdx.x;
  const int lane = tid & 31, wid = tid >> 5;
  const int fl = a.fl, fs = a.fs;
  const bool hann = (a.window == DSP_WIN_HANNING);

  #pragma unroll 1
  for (int j = tid; j < fl; j += kThreads) s_win[j] = a.win_f32[j];
  if (tid == 0) {
    mbar_init(s_bar, 1);
    mbar_fence_init();
    s_int[0] = (int)atomicAdd(a.work_counter, 1u);
  }
  __syncthreads();
  // de-phase the CTAs that share an SM: identical utterances make them run in lockstep otherwise,
  // so that their barrier / load bubbles coincide instead of filling one another
  if (a.stagger_ns > 0) {
    const unsigned wave = blockIdx.x / (unsigned)a.sm_count;
    if (wave > 0) { long long t0 = clock64(); const long long target = (long long)wave * a.stagger_ns * 2; while (clock64() - t0 < target) __nanosleep(200); }
  }

  // =========================================================================================
  // STATS WARPS: statistics + outputs of utterance i while the main warps work on utterance i+1
  // =========================================================================================
  if (wid >= kMainWarps) {
    const int sw = wid - kMainWarps;                       // owns sequences q with q % kStatsWarps == sw
    int* hist = s_hist + 256 * (1 + sw);
    float* cand = s_cand + 64 * (1 + sw);
    for (int it = 0;; ++it) {
      bar_sync(kBarFeatFull, kThreads);
      const int* mb = s_mail + 8 * (it & 1);
      const int u = mb[0], f2 = mb[1];
      if (u < 0) break;
      const int64_t fo = a.feat_offsets[u];
      float* stats = a.out.stats ? a.out.stats + (int64_t)u * kStats : nullptr;
      float st[5];
      if (f2 <= 32 * kStatsRegs) {
        // copy this warp's sequences to a per-lane array so the main warps can reuse the buffers at once
        float r[3][kStatsRegs];
#pragma unroll 1
        for (int q = sw; q < 3; q += kStatsWarps) {
          const float* src = q == 0 ? s_fe : (q == 1 ? s_fm : s_fz);
#pragma unroll 1
          for (int j = 0; j < kStatsRegs; ++j) { const int i = lane + 32 * j; r[q][j] = i < f2 ? src[i] : 0.f; }
        }
        bar_arrive(kBarFeatEmpty, kThreads);
#pragma unroll 1
        for (int q = sw; q < 3; q += kStatsWarps) {
          float* g = q == 0 ? a.out.energy : (q == 1 ? a.out.magnitude : a.out.zcr);
          if (g) {
#pragma unroll 1
            for (int j = 0; j < kStatsRegs; ++j) { const int i = lane + 32 * j; if (i < f2) g[fo + i] = r[q][j]; }
          }
          if (f2 > 0 && stats) {
            warp_sequence_stats(r[q], 1, f2, hist, cand, st);
            if (lane == 0) for (int k = 0; k < 5; ++k) stats[5 * q + k] = st[k];
          }
        }
      } else {
        // long sequences: work from shared memory, release the buffers afterwards
#pragma unroll 1
        for (int q = sw; q < 3; q += kStatsWarps) {
          const float* src = q == 0 ? s_fe : (q == 1 ? s_fm : s_fz);
          float* g = q == 0 ? a.out.energy : (q == 1 ? a.out.magnitude : a.out.zcr);
          for (int i = lane; i < f2; i += 32) if (g) g[fo + i] = src[i];
          if (stats) {
            warp_sequence_stats(src + lane, 32, f2, hist, cand, st);
            if (lane == 0) for (int k = 0; k < 5; ++k) stats[5 * q + k] = st[k];
          }
        }
        __syncwarp();
        bar_arrive(kBarFeatEmpty, kThreads);
      }
    }
    return;
  }

  // =========================================================================================
  // MAIN WARPS
  // =========================================================================================
  uint32_t parity = 0;
  (void)parity;
  __shared__ long long s_prof[16];
  long long t_prev = clock64();
  if (tid < 16) s_prof[tid] = 0;
  int u = s_int[0];
  int iter = 0;

  // window coefficients of the hop-128 / length-256 chain (P4 fast path): a lane owns samples
  // 8*(lane&15) .. +8 of every hop block; c = 0 is the first half of a frame, c = 1 the second
  const bool chain_cfg = (fs == 128 && fl == 256);
  float cw[2][8], cw2[2][8];
  if (chain_cfg) {
#pragma unroll
    for (int c = 0; c < 2; ++c)
#pragma unroll
      for (int q8 = 0; q8 < 8; ++q8) { const float w = s_win[c * 128 + 8 * (lane & 15) + q8]; cw[c][q8] = w; cw2[c][q8] = w * w; }
  }

  // issue the load of utterance `uu` (uniform over the main warps)
  auto issue_load = [&](int uu) {
    const int64_t off = a.offsets[uu];
    const int n = a.lengths ? a.lengths[uu] : (int)(a.offsets[uu + 1] - off);
    const int16_t* src = a.samples + off;
    const bool tma = ((reinterpret_cast<uintptr_t>(src) & 15) == 0);
    if (tma) {
      const uint32_t bytes = ((uint32_t)n * 2u) & ~15u;
      if (tid < 32) {
        if (bytes > 0) {
          if (tid == 0) { fence_proxy_async(); mbar_expect_tx(s_bar, bytes); }
          __syncwarp();
          const uint32_t chunk = (uint32_t)a.tma_chunk;
          for (uint32_t o = (uint32_t)tid * chunk; o < bytes; o += 32u * chunk) {
            const uint32_t sz = min(chunk, bytes - o);
            bulk_g2s(smem_u32(s_x) + o, reinterpret_cast<const unsigned char*>(src) + o, sz, s_bar);
          }
        }
      }
      // tail (< 8 samples) by plain loads
      const int done = (int)(bytes >> 1);
      if (tid >= 32 && tid < 32 + (n - done)) s_x[done + tid - 32] = src[done + tid - 32];
    } else if ((reinterpret_cast<uintptr_t>(src) & 3) == 0) {
      const uint32_t* s32 = reinterpret_cast<const uint32_t*>(src);
      uint32_t* d32 = reinterpret_cast<uint32_t*>(s_x);
      #pragma unroll 1
      for (int i = tid; i < (n >> 1); i += kMainThreads) d32[i] = __ldg(s32 + i);
      if ((n & 1) && tid == 0) s_x[n - 1] = src[n - 1];
    } else {
      #pragma unroll 1
      for (int i = tid; i < n; i += kMainThreads) s_x[i] = src[i];
    }
  };
  auto wait_load = [&](int uu) {
    const int64_t off = a.offsets[uu];
    const int n = a.lengths ? a.lengths[uu] : (int)(a.offsets[uu + 1] - off);
    const bool tma = ((reinterpret_cast<uintptr_t>(a.samples + off) & 15) == 0);
    if (tma && (((uint32_t)n * 2u) & ~15u) > 0) { mbar_wait_spin(s_bar, parity); parity ^= 1; }
    main_sync();
  };

  auto ld16 = [&](const void* p) -> int4 {
    if constexpr (kStream) return __ldg(reinterpret_cast<const int4*>(p));
    else return *reinterpret_cast<const int4*>(p);
  };

  if (!kStream && u < a.n_utts) issue_load(u);

  while (u < a.n_utts) {
    const int64_t off = a.offsets[u];
    const int n = a.lengths ? a.lengths[u] : (int)(a.offsets[u + 1] - off);
    const int16_t* x = kStream ? a.samples + off : s_x;
    if constexpr (kStream) {
      if (reinterpret_cast<uintptr_t>(x) & 15) {
        // misaligned start: not this kernel's layout -- hand the utterance to the float64 replay
        if (tid == kLeadTid) {
          const int slot = atomicAdd(a.flag_count, 1); a.flag_list[slot] = u;
          s_int[0] = (int)atomicAdd(a.work_counter, 1u);
        }
        main_sync();
        u = s_int[0];
        main_sync();
        continue;
      }
      main_sync();
    } else {
      wait_load(u);
    }
    if (tid == 0) s_int[0] = (int)atomicAdd(a.work_counter, 1u);   // next utterance, consumed after P4

    if (a.prof && tid == 0) { const long long t_ = clock64(); s_prof[0] += t_ - t_prev; t_prev = t_; }
    // =========================== P1: sum, min, max ===================================
    {
      int sum = 0;
      uint32_t mn2 = 0x7fff7fffu, mx2 = 0x80008000u;
      const int nvec = n >> 3;
      const int4* xv = reinterpret_cast<const int4*>(x);
      auto acc1 = [&](const int4& q) {
        sum = __dp2a_lo(q.x, 0x0101, sum); sum = __dp2a_lo(q.y, 0x0101, sum);
        sum = __dp2a_lo(q.z, 0x0101, sum); sum = __dp2a_lo(q.w, 0x0101, sum);
        mn2 = __vmins2(mn2, q.x); mx2 = __vmaxs2(mx2, q.x);
        mn2 = __vmins2(mn2, q.y); mx2 = __vmaxs2(mx2, q.y);
        mn2 = __vmins2(mn2, q.z); mx2 = __vmaxs2(mx2, q.z);
        mn2 = __vmins2(mn2, q.w); mx2 = __vmaxs2(mx2, q.w);
      };
      int v = tid;
      if constexpr (kStream) {
        for (; v + 3 * kMainThreads < nvec; v += 4 * kMainThreads) {     // 4 loads in flight per thread
          const int4 q0 = ld16(xv + v), q1 = ld16(xv + v + kMainThreads);
          const int4 q2 = ld16(xv + v + 2 * kMainThreads), q3 = ld16(xv + v + 3 * kMainThreads);
          acc1(q0); acc1(q1); acc1(q2); acc1(q3);
        }
      }
#pragma unroll 1
      for (; v < nvec; v += kMainThreads) { const int4 q = ld16(xv + v); acc1(q); }
      int mn = min(sext16(mn2), (int)mn2 >> 16), mx = max(sext16(mx2), (int)mx2 >> 16);
      if (tid < (n & 7)) { const int k = x[(nvec << 3) + tid]; sum += k; mn = min(mn, k); mx = max(mx, k); }
      // a thread's sum covers at most 2^20 / 96 samples (< 2^31 / 2^15), a warp's does not: a streaming build's warp
      // sees n / kMainWarps samples (up to 2^20 / 3), so the per-warp partials are 64-bit
      const long long wsum = warp_reduce((long long)sum, OpAddLL());
      mn = warp_reduce(mn, OpMinI());
      mx = warp_reduce(mx, OpMaxI());
      long long* part = reinterpret_cast<long long*>(s_sh);      // 3 * kWarps <= 27 values of the 64 in s_sh
      if (lane == 0) { part[wid] = wsum; part[kWarps + wid] = mn; part[2 * kWarps + wid] = mx; }
      main_sync();
      if (tid == kLeadTid) {
        long long S = 0; int gmn = 32767, gmx = -32768;
        #pragma unroll 1
        for (int w = 0; w < kMainWarps; ++w) { S += part[w]; gmn = min(gmn, (int)part[kWarps + w]); gmx = max(gmx, (int)part[2 * kWarps + w]); }
        const long long N = n > 0 ? n : 1;
        long long q = S / N; if ((S % N) != 0 && (S < 0)) --q;      // floor(S/N)
        const long long thr = q + 1;
        const long long R = S - N * thr;                             // in [-N, 0)
        const long long M = max(N * (long long)gmx - S, S - N * (long long)gmn);
        s_int[1] = (int)thr;
        s_dbl[0] = (double)R / (double)N;
        s_dbl[1] = (M > 0) ? (double)N / (double)M : 1.0;
        s_dbl[2] = (double)S / (double)N;
        s_int[3] = 0;   // flag
        s_int[4] = n;   // n3 (min)      -- initial values for the searches
        s_int[5] = -1;  // n4 (max)
      }
      main_sync();
    }
    UttConst uc;
    uc.thr = s_int[1]; uc.phi_d = s_dbl[0]; uc.phi = (float)uc.phi_d;
    uc.inv_m = s_dbl[1]; uc.mu = s_dbl[2];

    if (a.prof && tid == 0) { const long long t_ = clock64(); s_prof[1] += t_ - t_prev; t_prev = t_; }
    // the group-sum region doubles as the feature buffers the stats warps may still be reading
    if (iter > 0) bar_sync(kBarFeatEmpty, kThreads);

    if (a.prof && tid == 0) { const long long t_ = clock64(); s_prof[2] += t_ - t_prev; t_prev = t_; }
    // =========================== P2: group sums + sign bits ==========================
    const int ng = (n + kGroup - 1) / kGroup;
    {
      // resident mode: rotated vector order keeps the 16-byte shared-memory accesses conflict-free;
      // streaming mode reads its own 128-byte line through L1 and needs no rotation
      const int rot = kStream ? 0 : (tid & 7);               // == g & 7 for every group this thread owns
      for (int g = tid; g < ng; g += kMainThreads) {
        int s1 = 0;
        unsigned long long s2 = 0;
        uint32_t b0, b1;
        const int base = g * kGroup;
        if (base + kGroup <= n) {
          const unsigned char* gp = reinterpret_cast<const unsigned char*>(x + base);
          uint32_t nlo = 0, nhi = 0;         // "below the mean" bits, MSB-first, in processing order
          int s1b = 0;
          unsigned long long s2b = 0;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            // vectors j and j+4 of the (rotated) order feed two independent dependency chains
            const int4 qa = ld16(gp + 16 * ((j + rot) & 7));
            const int4 qb = ld16(gp + 16 * ((j + 4 + rot) & 7));
            const uint32_t wa[4] = {(uint32_t)qa.x, (uint32_t)qa.y, (uint32_t)qa.z, (uint32_t)qa.w};
            const uint32_t wb[4] = {(uint32_t)qb.x, (uint32_t)qb.y, (uint32_t)qb.z, (uint32_t)qb.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const int alo = sext16(wa[k]) - uc.thr, ahi = ((int)wa[k] >> 16) - uc.thr;
              const int blo = sext16(wb[k]) - uc.thr, bhi = ((int)wb[k] >> 16) - uc.thr;
              s1 += alo + ahi; s1b += blo + bhi;
              s2 += (unsigned long long)((long long)alo * alo) + (unsigned long long)((long long)ahi * ahi);
              s2b += (unsigned long long)((long long)blo * blo) + (unsigned long long)((long long)bhi * bhi);
              nhi = __funnelshift_l((uint32_t)alo, nhi, 1); nhi = __funnelshift_l((uint32_t)ahi, nhi, 1);
              nlo = __funnelshift_l((uint32_t)blo, nlo, 1); nlo = __funnelshift_l((uint32_t)bhi, nlo, 1);
            }
          }
          s1 += s1b; s2 += s2b;
          // stream (nhi:nlo) holds vector rot first (at the top); reverse to LSB-first, undo the rotation
          const unsigned long long y = ((unsigned long long)__brev(nlo) << 32) | (unsigned long long)__brev(nhi);
          const int sh = 8 * rot;
          const unsigned long long z = sh ? ((y << sh) | (y >> (64 - sh))) : y;
          b0 = ~(uint32_t)z; b1 = ~(uint32_t)(z >> 32);
        } else {
          b0 = 0; b1 = 0;
          #pragma unroll 1
          for (int i = 0; i < kGroup && base + i < n; ++i) {
            const int d = (int)x[base + i] - uc.thr;
            s1 += d; s2 += (unsigned long long)((long long)d * d);
            const uint32_t bit = (d >= 0);
            if (i < 32) b0 |= bit << i; else b1 |= bit << (i - 32);
          }
        }
        s_g1[g] = s1; s_g2[g] = s2;
        s_bits[2 * g] = b0; s_bits[2 * g + 1] = b1;
      }
    }
    if (tid < 4) s_bits[2 * ng + tid] = 0;
    main_sync();

    if (a.prof && tid == 0) { const long long t_ = clock64(); s_prof[3] += t_ - t_prev; t_prev = t_; }
    // =========================== P2b: EPD frame energies / crossings =================
    int f1 = 0;
    if (a.do_epd && n >= fl) f1 = (n - fl) / fs + 1;
    {
      double emx = 0.0, emn = INFINITY, amx = 0.0;
      for (int f = tid; f < f1; f += kMainThreads) {
        const int p = f * fs, q = p + fl;
        long long s1 = 0; unsigned long long s2 = 0;
        const int ga = (p + kGroup - 1) / kGroup, gb = q / kGroup;
        auto direct = [&](int i0, int i1) {
          #pragma unroll 1
          for (int i = i0; i < i1; ++i) { const int d = (int)x[i] - uc.thr; s1 += d; s2 += (unsigned long long)((long long)d * d); }
        };
        if (ga > gb) direct(p, q);
        else {
          for (int g = ga; g < gb; ++g) { s1 += s_g1[g]; s2 += s_g2[g]; }
          direct(p, ga * kGroup);
          direct(gb * kGroup, q);
        }
        // sum (d - phi)^2 from exact integer sums; `amx` bounds the rounding of the three terms
        const double t1 = 2.0 * uc.phi_d * (double)s1, t2 = (double)fl * uc.phi_d * uc.phi_d;
        const double ep = ((double)s2 - t1) + t2;
        const double e = ep * uc.inv_m * uc.inv_m;
        s_e[f] = e;
        s_z[f] = count_changes(s_bits, p, q);
        emx = fmax(emx, e); emn = fmin(emn, e);
        amx = fmax(amx, ((double)s2 + fabs(t1)) + t2);
      }
      emx = warp_reduce(emx, OpMaxD());
      emn = warp_reduce(emn, OpMinD());
      amx = warp_reduce(amx, OpMaxD());
      double* part = reinterpret_cast<double*>(s_sh);
      if (lane == 0) { part[wid] = emx; part[kWarps + wid] = amx; part[2 * kWarps + wid] = emn; }
      for (int i = tid; i < 256; i += kMainThreads) s_hist[i] = 0;     // first pass of the p90 select
      if (tid == 0) s_int[12 + 5] = 0;                                  // candidate counter
    }
    main_sync();

    if (a.prof && tid == 0) { const long long t_ = clock64(); s_prof[4] += t_ - t_prev; t_prev = t_; }
    // =========================== P3: endpoint decision ===============================
    int start = 0, end = n;
    if (f1 > 0) {
      // ---- 90th percentile: block-parallel radix select on float projections of E, first pass
      //      spread over [E_min, E_max]; the (<= 32) survivors are ranked in float64 by warp 0
      const double v = (double)(f1 - 1) * (90.0 / 100.0);
      const bool top = v >= (double)(f1 - 1);
      int* hist = s_hist;
      int* sel_state = s_int + 12;        // [0] lo  [1] shift  [2] rank  [3] cnt  [4] shift used  [5] cand count
      int* cand_idx = reinterpret_cast<int*>(s_cand);
      {
        // every thread derives the select state from the per-warp partials: no broadcast barrier
        const double* part = reinterpret_cast<const double*>(s_sh);
        double emx = 0.0, emn = INFINITY;
        #pragma unroll 1
        for (int w = 0; w < kMainWarps; ++w) { emx = fmax(emx, part[w]); emn = fmin(emn, part[2 * kWarps + w]); }
        const uint32_t kmin = __float_as_uint((float)emn), kmax = __float_as_uint((float)emx);
        if (tid == kLeadTid) {
          sel_state[0] = (int)kmin;
          sel_state[1] = first_shift(kmin, kmax);
          sel_state[2] = top ? f1 - 1 : (int)floor(v);
          sel_state[3] = f1;
          sel_state[4] = 32;
        }
        // noise floors (first/last min(5, F1/10) frames, :188-195, :241-247) by another warp meanwhile
        if (wid == (kMainWarps > 1 ? kLeadWarp - 1 : 0) && lane == 0) {
          const int nf = min(5, f1 / 10);
          double noise_e, noise_z;
          if (nf > 0) {
            double ve[10], vz[10];
            for (int i = 0; i < 2 * nf; ++i) {
              const int f = i < nf ? i : f1 - 2 * nf + i;
              ve[i] = s_e[f]; vz[i] = (double)s_z[f];
            }
            noise_e = noise_mean(ve, 2 * nf);
            noise_z = noise_mean(vz, 2 * nf);
          } else {
            noise_e = s_e[0]; noise_z = (double)s_z[0];
            #pragma unroll 1
            for (int i = 1; i < f1; ++i) { noise_e = fmin(noise_e, s_e[i]); noise_z = fmin(noise_z, (double)s_z[i]); }
          }
          s_dbl[8] = noise_e; s_dbl[9] = noise_z;
        }
        // first pass inline (histogram zeroed before the P2b barrier, state known to every thread)
        int pass_s = first_shift(kmin, kmax);
        uint32_t pass_lo = kmin;
        bool first = true;
        while (first ? f1 > 32 : sel_state[3] > 32) {
          if (!first) {
            pass_lo = (uint32_t)sel_state[0]; pass_s = sel_state[1];
            for (int i = tid; i < 256; i += kMainThreads) hist[i] = 0;
            main_sync();
          }
          #pragma unroll 1
          for (int f = tid; f < f1; f += kMainThreads) {
            const uint32_t k = __float_as_uint((float)s_e[f]);
            if (k >= pass_lo) { const uint32_t d = (k - pass_lo) >> pass_s; if (d < 256u) atomicAdd(&hist[d], 1); }
          }
          main_sync();
          if (wid == kLeadWarp) {
            int digit, rank, cnt;
            scan_bins(hist, lane, first ? (top ? f1 - 1 : (int)floor(v)) : sel_state[2], &digit, &rank, &cnt);
            __syncwarp();
            if (lane == 0) {
              sel_state[0] = (int)(pass_lo + ((uint32_t)digit << pass_s));
              sel_state[4] = pass_s;
              sel_state[2] = rank;
              sel_state[3] = (pass_s == 0 && cnt > 32) ? -cnt : cnt;     // negative: cannot be split further
              sel_state[1] = pass_s > 8 ? pass_s - 8 : 0;
            }
          }
          main_sync();
          first = false;
        }
        if (f1 <= 32) main_sync();      // publish sel_state / noise floors written above
      }
      if (a.prof && tid == 0) { const long long t_ = clock64(); s_prof[8] += t_ - t_prev; t_prev = t_; }
      {
        // gather the candidate frames of the final bin
        const uint32_t lo = (uint32_t)sel_state[0];
        const unsigned long long span = 1ull << sel_state[4];
        const bool all = f1 <= 32;
        #pragma unroll 1
        for (int f = tid; f < f1; f += kMainThreads) {
          const uint32_t k = __float_as_uint((float)s_e[f]);
          if (all || (k >= lo && (unsigned long long)(k - lo) < span)) {
            const int slot = atomicAdd(&sel_state[5], 1);
            if (slot < 32) cand_idx[slot] = f;
          }
        }
      }
      main_sync();
      if (a.prof && tid == 0) { const long long t_ = clock64(); s_prof[9] += t_ - t_prev; t_prev = t_; }
      if (wid == kLeadWarp) {
        int cnt = sel_state[3];
        const int rank = sel_state[2];
        bool unresolved = false;
        if (cnt < 0) { cnt = 32; unresolved = true; }     // > 32 frames share one float: replay in float64
        const double mine = lane < cnt ? s_e[cand_idx[lane]] : INFINITY;
        int below = 0;
        #pragma unroll 1
        for (int j = 0; j < cnt; ++j) {
          const double o = __shfl_sync(0xffffffffu, mine, j);
          below += (o < mine) || (o == mine && j < lane);
        }
        const int r1 = unresolved ? 0 : rank;
        const unsigned m1 = __ballot_sync(0xffffffffu, lane < cnt && below == r1);
        const unsigned m2 = __ballot_sync(0xffffffffu, lane < cnt && below == r1 + 1);
        const double ka = __shfl_sync(0xffffffffu, mine, __ffs(m1) - 1);
        double kb = m2 ? __shfl_sync(0xffffffffu, mine, __ffs(m2) - 1) : ka;
        if (!m2 && !top) {               // rank + 1 lies above the candidate bin
          const uint32_t lo = (uint32_t)sel_state[0];
          const unsigned long long span = 1ull << sel_state[4];
          double nxt = INFINITY;
          #pragma unroll 1
          for (int f = lane; f < f1; f += 32) {
            const double e = s_e[f];
            const uint32_t k = __float_as_uint((float)e);
            if (k >= lo && (unsigned long long)(k - lo) >= span) nxt = fmin(nxt, e);
          }
          nxt = warp_reduce(nxt, OpMinD());
          kb = nxt == INFINITY ? ka : nxt;
        }
        if (top) kb = ka;
        if (lane == 0) {
          const double* part = reinterpret_cast<const double*>(s_sh);
          double emx = 0.0, amx = 0.0;
          #pragma unroll 1
          for (int w = 0; w < kMainWarps; ++w) { emx = fmax(emx, part[w]); amx = fmax(amx, part[kWarps + w]); }
          const double speech = np_lerp(ka, kb, v - floor(v));
          const double noise_e = s_dbl[8], noise_z = s_dbl[9];
          const double t1 = speech * a.hr;
          const double t2 = noise_e + (speech - noise_e) * a.lr;
          const double t3 = noise_z * a.zr;
          s_dbl[3] = t1; s_dbl[4] = t2; s_dbl[5] = t3;
          // Slack on the thresholds (DESIGN.md "numerics"): 2^-40 relative, the rounding of our own
          // three-term energy formula at its largest magnitude, and the reference's mean-rounding
          // term |mu| * sqrt(fl * E) / m at E_max, each with a >= 4x margin.
          const double eps = 1.0 / 1099511627776.0;  // 2^-40
          // sqrt(y) <= (y + 1) / 2: an upper bound is all a slack needs
          const double smax = 8.881784197001252e-16 /* 2^-50 */ *
                              (fabs(uc.mu) * 0.5 * ((double)fl * emx + 1.0) * uc.inv_m + amx * uc.inv_m * uc.inv_m);
          const double tol1 = eps * fabs(t1) + fabs(a.hr) * smax;
          const double tol2 = eps * (fabs(noise_e) + fabs(a.lr) * (fabs(speech) + fabs(noise_e))) +
                              (fabs(1.0 - a.lr) + fabs(a.lr)) * smax;
          s_dbl[6] = tol1 + smax + eps * emx;      // per-frame slack bounded at its utterance maximum
          s_dbl[7] = tol2 + smax + eps * emx;
          s_int[6] = 0; s_int[7] = f1 - 1; s_int[8] = 0; s_int[9] = f1 - 1;
          if (unresolved) s_int[3] = 1;
        }
      }
      main_sync();
      if (a.prof && tid == 0) { const long long t_ = clock64(); s_prof[10] += t_ - t_prev; t_prev = t_; }
      const double t1 = s_dbl[3], t2 = s_dbl[4], t3 = s_dbl[5];
      const double tol1 = s_dbl[6], tol2 = s_dbl[7];
      {
        int n3 = f1, n4 = -1, flag = 0;
        for (int f = tid; f < f1; f += kMainThreads) {
          const double e = s_e[f];
          if (e > t1) { n3 = min(n3, f); n4 = max(n4, f); }
          if (fabs(e - t1) <= tol1 && !(e == 0.0 && t1 == 0.0)) flag = 1;
          if (fabs(e - t2) <= tol2 && !(e == 0.0 && t2 == 0.0)) flag = 1;
        }
        n3 = warp_reduce(n3, OpMinI()); n4 = warp_reduce(n4, OpMaxI());
        flag = warp_reduce(flag, OpMaxI());
        if (lane == 0) {
          if (n3 < f1) atomicMin(&s_int[4], n3);
          if (n4 >= 0) atomicMax(&s_int[5], n4);
          if (flag) atomicOr(&s_int[3], 1);
        }
      }
      main_sync();
      if (a.prof && tid == 0) { const long long t_ = clock64(); s_prof[11] += t_ - t_prev; t_prev = t_; }
      const int n3 = s_int[4], n4 = s_int[5];
      if (n4 >= 0) {
        {
          int n2 = 0, n5 = f1 - 1;
          for (int f = tid; f < f1; f += kMainThreads)
            if (s_e[f] <= t2) { if (f < n3) n2 = max(n2, f + 1); if (f > n4) n5 = min(n5, f - 1); }
          n2 = warp_reduce(n2, OpMaxI()); n5 = warp_reduce(n5, OpMinI());
          if (lane == 0) { if (n2 > 0) atomicMax(&s_int[6], n2); if (n5 < f1 - 1) atomicMin(&s_int[7], n5); }
        }
        main_sync();
        const int n2 = s_int[6], n5 = s_int[7];
        {
          int n1 = 0, n6 = f1 - 1;
          for (int f = tid; f < f1; f += kMainThreads)
            if ((double)s_z[f] <= t3) { if (f < n2) n1 = max(n1, f + 1); if (f > n5) n6 = min(n6, f - 1); }
          n1 = warp_reduce(n1, OpMaxI()); n6 = warp_reduce(n6, OpMinI());
          if (lane == 0) { if (n1 > 0) atomicMax(&s_int[8], n1); if (n6 < f1 - 1) atomicMin(&s_int[9], n6); }
        }
        main_sync();
        start = s_int[8] * fs;
        end = min(s_int[9] * fs + fl, n);
      }
      // EPD lists out (the group-sum region is dead from here on; E/Z stay valid)
      if (a.out.epd_energy || a.out.epd_zcr) {
        const int64_t eo = a.epd_offsets[u];
        #pragma unroll 1
        for (int f = tid; f < f1; f += kMainThreads) {
          if (a.out.epd_energy) a.out.epd_energy[eo + f] = s_e[f];
          if (a.out.epd_zcr) a.out.epd_zcr[eo + f] = (float)s_z[f];
        }
      }
    }
    if (a.prof && tid == 0) { const long long t_ = clock64(); s_prof[5] += t_ - t_prev; t_prev = t_; }
    const int flagged = s_int[3];

    // =========================== P4: windowed frame features =========================
    const int seg = end - start;
    const int f2 = (int)frame_count_host_device(seg, fl, fs);
    int f2_chain = 0;      // frames [0, f2_chain) done by the chain path, the rest generically
    if (chain_cfg && (start & 127) == 0 && seg >= 256) f2_chain = (seg - 256) / 128 + 1;
    if (f2_chain > f2) f2_chain = f2;
    if (f2_chain > 0) {
      // 16 lanes per chain; a chain covers `per` consecutive frames = per + 1 hop blocks.
      constexpr int kChains = kMainThreads / 16;
      const int chain = tid >> 4, sub = tid & 15;
      const int per = (f2_chain + kChains - 1) / kChains;
      const int fa = chain * per, fb = min(fa + per, f2_chain);
      const float phi = uc.phi;
      float ce = 0.f, cm = 0.f;                       // first-half partials of the previous block
      const bool hi8 = (sub & 8) != 0;
      int4 qn = make_int4(0, 0, 0, 0);
      if (kStream && fa < fb) qn = ld16(x + start + fa * 128 + 8 * sub);
      for (int i = 0; i <= per; ++i) {             // uniform trip count: the shuffles below are warp-wide
        const int b = fa + i;
        const bool live = (fa < fb) && (b <= fb);
        int4 q = qn;
        if constexpr (kStream) {                   // global loads: fetch the next block one step ahead
          if ((fa < fb) && (b + 1 <= fb)) qn = ld16(x + start + (b + 1) * 128 + 8 * sub);
        } else {
          if (live) q = ld16(x + start + b * 128 + 8 * sub);
        }
        const uint32_t w[4] = {(uint32_t)q.x, (uint32_t)q.y, (uint32_t)q.z, (uint32_t)q.w};
        float e0 = 0.f, m0 = 0.f, e1 = ce, m1 = cm;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float dlo = (float)(sext16(w[k]) - uc.thr) - phi;
          const float dhi = (float)(((int)w[k] >> 16) - uc.thr) - phi;
          const float qlo = dlo * dlo, qhi = dhi * dhi;
          const float alo = fabsf(dlo), ahi = fabsf(dhi);
          e0 = fmaf(cw2[0][2 * k], qlo, e0); m0 = fmaf(cw[0][2 * k], alo, m0);
          e1 = fmaf(cw2[1][2 * k], qlo, e1); m1 = fmaf(cw[1][2 * k], alo, m1);
          e0 = fmaf(cw2[0][2 * k + 1], qhi, e0); m0 = fmaf(cw[0][2 * k + 1], ahi, m0);
          e1 = fmaf(cw2[1][2 * k + 1], qhi, e1); m1 = fmaf(cw[1][2 * k + 1], ahi, m1);
        }
        ce = e0; cm = m0;
        // frame b-1 = first half carried from the previous block (in e1/m1 through ce/cm) + this
        // block as its second half: transposed reduction of (e1, m1) over the chain's 16 lanes
        const float send = hi8 ? e1 : m1, keep = hi8 ? m1 : e1;
        float vv = keep + __shfl_xor_sync(0xffffffffu, send, 8);
        vv += __shfl_xor_sync(0xffffffffu, vv, 4);
        vv += __shfl_xor_sync(0xffffffffu, vv, 2);
        vv += __shfl_xor_sync(0xffffffffu, vv, 1);
        if (live && b > fa && (sub & 7) == 0) (hi8 ? s_fm : s_fe)[b - 1] = vv;    // raw sums, scaled below
      }
    }
    if (f2_chain < f2) {
      const int sub = tid & (kLanesPerFrame - 1);
      const int slot = tid / kLanesPerFrame;
      constexpr int kSlots = kMainThreads / kLanesPerFrame;
      const bool vec_ok = ((start & 7) == 0) && ((fs & 7) == 0);
      const float phi = uc.phi;
      for (int t0 = f2_chain; t0 < f2; t0 += kSlots) {
        const int t = t0 + slot;
        float e = 0.f, m = 0.f;
        int p = 0, valid = 0;
        if (t < f2) {
          p = start + t * fs;
          valid = min(fl, end - p);
          int jdone = 0;
          if (vec_ok) {
            const int nv = valid >> 3;
            const int4* xv = reinterpret_cast<const int4*>(x + p);
            const float4* wv = reinterpret_cast<const float4*>(s_win);
            for (int vq = sub; vq < nv; vq += kLanesPerFrame) {
              const int4 q = ld16(xv + vq);
              const float4 wa = wv[2 * vq], wb = wv[2 * vq + 1];
              const uint32_t w[4] = {(uint32_t)q.x, (uint32_t)q.y, (uint32_t)q.z, (uint32_t)q.w};
              const float ww[8] = {wa.x, wa.y, wa.z, wa.w, wb.x, wb.y, wb.z, wb.w};
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const float dlo = (float)(sext16(w[k]) - uc.thr) - phi;
                const float dhi = (float)(((int)w[k] >> 16) - uc.thr) - phi;
                const float alo = ww[2 * k] * dlo, ahi = ww[2 * k + 1] * dhi;
                e = fmaf(alo, alo, e); m += fabsf(alo);
                e = fmaf(ahi, ahi, e); m += fabsf(ahi);
              }
            }
            jdone = nv << 3;
          }
          #pragma unroll 1
          for (int j = jdone + sub; j < valid; j += kLanesPerFrame) {
            const float d = (float)((int)x[p + j] - uc.thr) - phi;
            const float av = s_win[j] * d;
            e = fmaf(av, av, e); m += fabsf(av);
          }
        }
#pragma unroll
        for (int o = kLanesPerFrame / 2; o > 0; o >>= 1) {
          e += __shfl_xor_sync(0xffffffffu, e, o);
          m += __shfl_xor_sync(0xffffffffu, m, o);
        }
        if (t < f2 && sub == 0) { s_fe[t] = e; s_fm[t] = m; }                      // raw sums, scaled below
      }
    }
    main_sync();
    if (a.prof && tid == 0) { const long long t_ = clock64(); s_prof[6] += t_ - t_prev; t_prev = t_; }
    // peak normalisation (1/m^2, 1/m) and zero crossings, one frame per thread.  A full frame of
    // the trimmed segment IS an endpoint-detection frame (start is a multiple of the hop), so its
    // crossing count is already in s_z; only Hanning's zeroed end points need patching.
    #pragma unroll 1
    for (int t = tid; t < f2; t += kMainThreads) {
      const int p = start + t * fs;
      const int valid = min(fl, end - p);
      s_fe[t] = (float)((double)s_fe[t] * uc.inv_m * uc.inv_m);
      s_fm[t] = (float)((double)s_fm[t] * uc.inv_m);
      int zc;
      if (f1 > 0 && valid == fl && !(hann && fl <= 2)) {
        zc = s_z[p / fs];
        if (hann) {
          const int s0 = bit_at(s_bits, p), s1 = bit_at(s_bits, p + 1);
          const int sl = bit_at(s_bits, p + fl - 1), sp = bit_at(s_bits, p + fl - 2);
          zc += (s1 - (s0 ^ s1)) + (sp - (sp ^ sl));
        }
      } else {
        zc = frame_zcr(s_bits, p, valid, fl, hann);
      }
      s_fz[t] = (float)zc;
    }
    // per-utterance scalars, mailbox for the stats warps
    if (tid == 0) {
      int status = DSP_UTT_OK;
      if (seg <= 0) status = DSP_UTT_EMPTY; else if (f2 == 0) status = DSP_UTT_NO_FRAMES;
      if (a.out.start) a.out.start[u] = start;
      if (a.out.end) a.out.end[u] = end;
      if (a.out.n_epd_frames) a.out.n_epd_frames[u] = f1;
      if (a.out.n_frames) a.out.n_frames[u] = f2;
      if (a.out.status) a.out.status[u] = status;
      if (flagged) { const int slot = atomicAdd(a.flag_count, 1); a.flag_list[slot] = u; }
      int* mb = s_mail + 8 * (iter & 1);
      mb[0] = u; mb[1] = f2;
    }
    main_sync();   // samples / sign bits are dead, features + mailbox are complete
    bar_arrive(kBarFeatFull, kThreads);

    if (a.prof && tid == 0) { const long long t_ = clock64(); s_prof[7] += t_ - t_prev; t_prev = t_; }
    const int u_next = s_int[0];
    if (!kStream && u_next < a.n_utts) issue_load(u_next);
    u = u_next;
    ++iter;
  }
  if (a.prof && tid == 0) { for (int i = 0; i < 12; ++i) atomicAdd((unsigned long long*)&a.prof[i], (unsigned long long)s_prof[i]); atomicAdd((unsigned long long*)&a.prof[15], (unsigned long long)iter); }
  // tell the stats warps to stop
  if (iter > 0) bar_sync(kBarFeatEmpty, kThreads);
  if (tid == 0) s_mail[8 * (iter & 1)] = -1;
  main_sync();
  bar_arrive(kBarFeatFull, kThreads);
}

namespace {
using PcmKernel = void (*)(const PcmArgs);
struct Variant { PcmKernel fn; int threads; bool stream; };
// [0], [8] and [9] are shared-memory-resident builds (any alignment); the rest are streaming builds
const Variant kVariants[] = {
    {frontend_pcm_kernel<false, 256, 2, 2>, 256, false},
    {frontend_pcm_kernel<true, 128, 1, 4>, 128, true},
    {frontend_pcm_kernel<true, 128, 1, 5>, 128, true},
    {frontend_pcm_kernel<true, 128, 1, 6>, 128, true},
    {frontend_pcm_kernel<true, 256, 2, 2>, 256, true},
    {frontend_pcm_kernel<true, 256, 2, 3>, 256, true},
    {frontend_pcm_kernel<true, 192, 2, 4>, 192, true},
    {frontend_pcm_kernel<true, 160, 1, 4>, 160, true},
    {frontend_pcm_kernel<false, 256, 1, 2>, 256, false},
    {frontend_pcm_kernel<false, 288, 1, 2>, 288, false},
};
constexpr int kNumVariants = (int)(sizeof(kVariants) / sizeof(kVariants[0]));
}  // namespace

int pcm_num_variants() { return kNumVariants; }
bool pcm_variant_streams(int v) { return kVariants[v].stream; }

cudaError_t launch_frontend_pcm(int variant, const PcmArgs& a, int grid, size_t smem, cudaStream_t st) {
  const Variant& v = kVariants[variant];
  cudaError_t e = cudaFuncSetAttribute(v.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  v.fn<<<grid, v.threads, smem, st>>>(a);
  return cudaGetLastError();
}

int pcm_kernel_max_ctas_per_sm(int variant, size_t smem, size_t smem_optin) {
  const Variant& v = kVariants[variant];
  cudaFuncAttributes fa{};
  int n = 0;
  // the kernel's static shared memory (s_prof) counts against the opt-in per-block maximum too
  if (cudaFuncGetAttributes(&fa, v.fn) != cudaSuccess || fa.sharedSizeBytes + smem > smem_optin) return 0;
  if (cudaFuncSetAttribute(v.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
    cudaGetLastError();      // a refused size means "does not fit", not an error for the next launch to report
    return 0;
  }
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, v.fn, v.threads, smem) != cudaSuccess) return 0;
  return n;
}

}  // namespace dsp
