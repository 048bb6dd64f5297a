// Pipelined fused front-end kernel for 16-bit mono PCM (the throughput path, round-1 redesign).
//
// One persistent CTA per SM, three warp roles that never meet at a CTA-wide barrier:
//
//   control warp (1)   dynamic utterance scheduler + TMA producer.  Utterances are cut into 4 KB
//                      chunks that travel through a ring of shared-memory slots (full/empty
//                      mbarrier pair per slot, cp.async.bulk), so the next utterances are in
//                      flight while the current one is being reduced.
//   stream warps (8)   the two passes that touch EVERY sample, straight from the ring:
//                        A  per 64-sample group: sum k, sum k^2 (exact integers via dp4a on the
//                           byte planes), min, max                  -> DC (rational S/N), peak
//                        B  one sign bit per sample (k >= thr, thr = floor(S/N)+1)
//                        F  every endpoint-detection frame from the group sums / sign bits:
//                           float64 energy, zero-crossing count  -> a small per-utterance record
//                      The ring slots are released right after pass B: samples stay on chip for
//                      exactly two reads and HBM is read once.
//   tail warps (<= 7)  one WARP per utterance, several utterances in flight: 90th percentile by
//                      bisection on float keys + float64 ranking of <= 32 survivors, thresholds
//                      in NumPy's order, the six endpoint searches (certified margins, else
//                      float64 replay), windowed energy / magnitude of the trimmed segment (re-read
//                      from L2, fp32), the 15 statistics, all outputs.  Purely warp-synchronous:
//                      its latency is hidden by the other tail warps and the stream warps.
//
// Exactness argument: identical to frontend_pcm.cu (DESIGN.md "numerics"); only the schedule differs.
// Reference: src/audio_processing.py:49-90,135-275,299-333; src/feature_extraction.py:12-88.
#include <algorithm>
#include "kernels.cuh"
#include "ptx.cuh"

namespace dsp {

namespace {

constexpr int kGroup = 64;                 // samples per group-sum record
constexpr int kChunkSamples = 2048;        // samples per ring slot
constexpr int kChunkBytes = 2 * kChunkSamples;
constexpr int kGroupsPerChunk = kChunkSamples / kGroup;   // 32: one group per stream lane
#ifndef DSP_PIPE_STREAM_WARPS
#define DSP_PIPE_STREAM_WARPS 8
#endif
// 8 stream warps (512 threads, 128 registers each) measure best with the batch hand-off below: 3.12 ms per 100k
// utterances against 3.26 (12 warps), 3.69 (16) and 3.57 (4) -- every stream warp repeats ~140 instructions of
// per-utterance set-up, and 22 chunks split 3/3/3/3/3/3/2/2 over 8 warps.  More than 8 use the register split.
constexpr int kStreamWarps = DSP_PIPE_STREAM_WARPS;       // a multiple of 4: whole warpgroups (setmaxnreg)
#ifndef DSP_PIPE_TAIL_WARPS
#define DSP_PIPE_TAIL_WARPS 7
#endif
// 7 tail warps: with 11 (-DDSP_PIPE_TAIL_WARPS=11 -DDSP_PIPE_STREAM_REGS=72: 640 threads, stream warps at 72 and tail warps at
// 112 registers, 22 records, a 24-slot ring) the kernel is parity-green and slower, 3.81 against 3.43 ms per 100k utterances
constexpr int kMaxTailWarps = DSP_PIPE_TAIL_WARPS;        // tail warps + the control warp: whole warpgroups too
constexpr int kPipeWarps = kStreamWarps + kMaxTailWarps + 1;
constexpr int kPipeThreads = 32 * kPipeWarps;             // 512
// Register split (setmaxnreg, per warpgroup; only for kStreamWarps > 8): the stream warps run short integer loops and give their
// registers to the tail warps, which keep whole sequences in registers.  The launch allocates
// kLaunchRegs = 65536 / kPipeThreads registers per thread (rounded down to 8) and the CTA owns only those:
// setmaxnreg.inc can take no more than the stream warps have given back, or it waits forever.
constexpr bool kSplitRegs = kPipeWarps > 16;              // more than 512 threads: 128 registers each no longer fit
constexpr int kLaunchRegs = (65536 / kPipeThreads) & ~7;
#ifndef DSP_PIPE_STREAM_REGS
#define DSP_PIPE_STREAM_REGS (DSP_PIPE_STREAM_WARPS == 16 ? 56 : 64)
#endif
constexpr int kStreamRegs = DSP_PIPE_STREAM_REGS;
constexpr int kTailRegs = ((kLaunchRegs * kPipeThreads - kStreamWarps * 32 * kStreamRegs) / ((kMaxTailWarps + 1) * 32)) & ~7;
static_assert(kStreamWarps % 4 == 0 && (kMaxTailWarps + 1) % 4 == 0, "roles must cover whole warpgroups");
static_assert(!kSplitRegs || kStreamWarps * 32 * kStreamRegs + (kMaxTailWarps + 1) * 32 * kTailRegs <= kLaunchRegs * kPipeThreads, "register pool of the CTA");
static_assert(!kSplitRegs || kTailRegs >= 104, "tail warps keep whole sequences in registers");
constexpr int kStreamThreads = 32 * kStreamWarps;
constexpr int kDescRing = 64;              // > max ring slots: the producer can never lap a reader
constexpr int kMaxRingSlots = 56;
constexpr int kRecHdr = 128;
// EPD frames per lane whose float keys stay in registers: 416 frames = 1.2 s at 256 / 128 for the specialised instantiation
// (its code size is what its speed hangs on), 704 frames for the general one (1 s at a hop of 64)
template <bool kChain> constexpr int key_regs() { return kChain ? 13 : 22; }
constexpr int kLanesPerFrame = 8;          // generic windowed pass: lanes cooperating on one frame

// per-group record of pass B (s_meta): bits 0-6 sign changes inside the group, then the sign bits of its samples
// 0,2,4,6,8 (kMetaE), 1,3,5,7 (kMetaO), 62 (kMetaP) and 63 (kMetaL)
constexpr int kMetaE = 8, kMetaO = 13, kMetaP = 17, kMetaL = 18;
__host__ __device__ constexpr int meta_bit(int i) { return (i & 1) ? kMetaO + (i >> 1) : kMetaE + (i >> 1); }

constexpr int kBarStream = 1;              // named barrier of the stream warps
// record hand-offs use named barriers too (a warp parked on bar.sync costs no issue slots, a warp polling an
// mbarrier does): kBarRecFull + r is "record r is complete" (stream warps arrive, its tail warp syncs),
// kBarRecEmpty + r is "record r is free again" (the tail warp arrives, the stream warps sync)
constexpr int kBarRecFull = 2, kBarRecEmpty = 9;
constexpr int kRecBarThreads = 32 * (kStreamWarps + 1);   // the stream warps + the record's tail warp
// Batch mode: records are handed over kBatch at a time (one per tail warp), double-buffered: the stream warps arrive on
// kBarBatchFull + b after the last record of batch b, ALL tail warps sync on it and therefore run decision / window /
// statistics at the same time -- one walk through the tail's ~25 KB of code then serves kBatch utterances instead of one
// (the instruction-miss path, gcc, runs at 94 % of its peak with staggered tail warps).  kBarBatchEmpty + b: the tail
// warps arrive when they are done with batch b, the stream warps sync before they refill it.
#ifndef DSP_PIPE_BATCH
#define DSP_PIPE_BATCH 1
#endif
#ifndef DSP_CHAIN_PACKED
#define DSP_CHAIN_PACKED 1          // window chain on packed fp32x2 arithmetic (0: the scalar FFMA build)
#endif
constexpr bool kBatchMode = DSP_PIPE_BATCH != 0;
constexpr int kBatch = kMaxTailWarps;
constexpr int kBarBatchFull = 2, kBarBatchEmpty = 4;
constexpr int kBatchBarThreads = 32 * (kStreamWarps + kMaxTailWarps);

struct PipeLayout {
  int ring, gsum, head, bits, meta, rec, scratch, win, desc, part, consts, bars, total;
  int rec_bytes, rec_e, rec_fe, rec_fm, rec_z, rec_zf;
};

__host__ __device__ inline int al16(int x) { return (x + 15) & ~15; }

// R ring slots, capG groups / capF frames per utterance, nrec records (= active tail warps)
__host__ __device__ inline PipeLayout make_pipe_layout(int R, int capG, int capF, int fl, int nrec) {
  PipeLayout L;
  int o = 0;
  L.ring = o;    o += R * kChunkBytes;
  L.gsum = o;    o += 2 * 8 * capG;
  L.head = o;    o += 2 * 8 * capG;
  L.bits = o;    o += al16(8 * capG + 16);
  L.meta = o;    o += al16(4 * capG);
  L.rec_e = kRecHdr;
  L.rec_fe = L.rec_e;                       // the feature sequences reuse the (dead) energy array
  L.rec_fm = L.rec_e + 4 * capF;
  L.rec_z = L.rec_e + al16(8 * capF);
  L.rec_zf = L.rec_z + al16(2 * capF);
  L.rec_bytes = L.rec_zf + al16(2 * capF);
  L.rec = o;     o += nrec * L.rec_bytes;
  L.scratch = o; o += nrec * 256;
  L.win = o;     o += al16(4 * fl);
  L.desc = o;    o += kDescRing * 8;
  L.part = o;    o += 2 * kStreamWarps * 16;
  L.consts = o;  o += 2 * 64;
  L.bars = o;    o += 8 * (2 * R + 2 * nrec);
  L.total = o;
  return L;
}

// ---- integer dot products on byte planes ------------------------------------------------
__device__ __forceinline__ int dp4a_ss(int a, int b, int c) { int d; asm("dp4a.s32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c)); return d; }
__device__ __forceinline__ int dp4a_su(int a, uint32_t b, int c) { int d; asm("dp4a.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c)); return d; }
__device__ __forceinline__ uint32_t dp4a_uu(uint32_t a, uint32_t b, uint32_t c) { uint32_t d; asm("dp4a.u32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c)); return d; }

// ---- packed fp32x2 arithmetic (sm_100: FFMA2 / FADD2 / FMUL2) ---------------------------------
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pk2(float a, float b) { f32x2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ float hsum2(f32x2 v) { float a, b; asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); return a + b; }
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) { f32x2 d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) { f32x2 d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) { f32x2 d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }

// frame_signal's frame count (kernels.cuh frame_count_host_device) in 32-bit arithmetic
__device__ __forceinline__ int frame_count32(int n, int fl, int fs) {
  if (n <= 0) return 0;
  const int a = (n + fs - 1) / fs;
  const int rem = n > fl ? n - fl : 0;
  const int b = (rem + fs - 1) / fs + 1;
  return a < b ? a : b;
}

// ---- sign-bit string helpers ---------------------------------------------------------------------------------------
// The string is kept in the form pass B produces it in: per 64-sample group two 32-bit planes, E (bit a = sample 2a is
// above the mean) at bits[2g] and O (sample 2a + 1) at bits[2g + 1].  Sign changes at the pairs (i, i + 1) of a group:
// even i = 2a are the bits of E ^ O, odd i = 2a + 1 the bits of O ^ (E shifted down by one, the next group's first
// sample moving into bit 31).  Nothing has to interleave the planes: pass B keeps its 2-instructions-per-word form for
// the ragged-edge geometries too, and a count over a range costs what it cost on the linear string.
__device__ __forceinline__ int bit_at(const uint32_t* bits, int i) { return (bits[2 * (i >> 6) + (i & 1)] >> ((i & 63) >> 1)) & 1; }
__device__ __forceinline__ uint32_t low_mask(int n) { return n >= 32 ? 0xffffffffu : ((1u << n) - 1u); }

// sign changes at the pairs (i, i + 1), i in [p, q - 2] (stream positions)
__device__ __forceinline__ int count_changes(const uint32_t* bits, int p, int q) {
  if (q - p < 2) return 0;
  const int last = q - 2;
  const int g0 = p >> 6, g1 = last >> 6;
  const int lo = p & 63, hi = (last & 63) + 1;                 // pairs lo.. of the first group, ..hi-1 of the last
  const uint32_t mE0 = ~low_mask((lo + 1) >> 1), mO0 = ~low_mask(lo >> 1);
  const uint32_t mE1 = low_mask((hi + 1) >> 1), mO1 = low_mask(hi >> 1);
  uint32_t E = bits[2 * g0], O = bits[2 * g0 + 1], En = bits[2 * g0 + 2];
  uint32_t x1 = E ^ O, x2 = O ^ __funnelshift_r(E, En, 1);
  if (g0 == g1) return __popc(x1 & mE0 & mE1) + __popc(x2 & mO0 & mO1);
  int c = __popc(x1 & mE0) + __popc(x2 & mO0);
  // (two groups per trip, their loads independent: this loop is on the critical path of the ragged geometries' pass F,
  //  where a thread walks the ~9 groups of its half of a frame by itself)
  int g = g0 + 1;
#pragma unroll 1
  for (; g + 1 < g1; g += 2) {
    const uint32_t Ea = En, Oa = bits[2 * g + 1], Eb = bits[2 * g + 2], Ob = bits[2 * g + 3], Ec = bits[2 * g + 4];
    c += __popc(Ea ^ Oa) + __popc(Oa ^ __funnelshift_r(Ea, Eb, 1)) + __popc(Eb ^ Ob) + __popc(Ob ^ __funnelshift_r(Eb, Ec, 1));
    En = Ec;
  }
#pragma unroll 1
  for (; g < g1; ++g) {
    E = En; O = bits[2 * g + 1]; En = bits[2 * g + 2];
    c += __popc(E ^ O) + __popc(O ^ __funnelshift_r(E, En, 1));
  }
  E = En; O = bits[2 * g1 + 1]; En = bits[2 * g1 + 2];
  c += __popc((E ^ O) & mE1) + __popc((O ^ __funnelshift_r(E, En, 1)) & mO1);
  return c;
}

// zero crossings of one windowed frame (compute_zero_crossing_rate on frame*window,
// audio_processing.py:119-132): zero padding and Hanning's exact-zero end points count as negative
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

__device__ __forceinline__ double warp_min_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_min_f(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// ---------------------------------------------------------------------------------------
// Statistics of one non-negative float sequence by ONE warp (compute_statistics,
// feature_extraction.py:46-62): mean, population std, max, min, and the median by bisection on
// the float bit patterns (no shared-memory histogram: a tail warp owns nothing but its record).
// get(i) yields element i.
// ---------------------------------------------------------------------------------------
template <class Get>
__device__ __forceinline__ void warp_stats(Get get, int n, float* out5) {
  const int lane = threadIdx.x & 31;
  double sum = 0.0;
  uint32_t kmx = 0u, kmn = 0xffffffffu;
#pragma unroll 1
  for (int i = lane; i < n; i += 32) { const float x = get(i); sum += (double)x; const uint32_t k = __float_as_uint(x); kmx = max(kmx, k); kmn = min(kmn, k); }
  sum = warp_reduce(sum, OpAddD());
  kmx = __reduce_max_sync(0xffffffffu, kmx);
  kmn = __reduce_min_sync(0xffffffffu, kmn);
  const double mean = sum / (double)n;
  double ss = 0.0;
#pragma unroll 1
  for (int i = lane; i < n; i += 32) { const double d = (double)get(i) - mean; ss += d * d; }
  ss = warp_reduce(ss, OpAddD());
  // median: key of rank r = (n-1)/2 by bisection; rank r+1 is the same key or the next larger one
  const int rank = (n - 1) >> 1;
  uint32_t prefix = kmn;
  const uint32_t diff = kmn ^ kmx;
  if (diff) {
    int b = 31 - __clz(diff);
    prefix = kmn & ~((2u << b) - 1u);
    int cnt_lo = 0, cnt_bin = n;
    while (b >= 0 && cnt_bin > 1) {
      const uint32_t trial = prefix | (1u << b);
      int c = 0;
#pragma unroll 1
      for (int i = lane; i < n; i += 32) c += (__float_as_uint(get(i)) < trial);
      c = __reduce_add_sync(0xffffffffu, c);
      if (rank < c) cnt_bin = c - cnt_lo;
      else { prefix = trial; cnt_bin = cnt_lo + cnt_bin - c; cnt_lo = c; }
      --b;
    }
    if (b >= 0) {      // a single key is left in [prefix, prefix + 2^(b+1)): fetch it
      const uint32_t hi = prefix + ((2u << b) - 1u);
      uint32_t k = 0xffffffffu;
#pragma unroll 1
      for (int i = lane; i < n; i += 32) { const uint32_t kk = __float_as_uint(get(i)); if (kk >= prefix && kk <= hi) k = min(k, kk); }
      prefix = __reduce_min_sync(0xffffffffu, k);
    }
  }
  const float sel = __uint_as_float(prefix);
  float sel2 = sel;
  if (!(n & 1)) {
    int le = 0;
    uint32_t nxt = 0xffffffffu;
#pragma unroll 1
    for (int i = lane; i < n; i += 32) { const uint32_t kk = __float_as_uint(get(i)); if (kk <= prefix) ++le; else nxt = min(nxt, kk); }
    le = __reduce_add_sync(0xffffffffu, le);
    nxt = __reduce_min_sync(0xffffffffu, nxt);
    if (le < rank + 2 && nxt != 0xffffffffu) sel2 = __uint_as_float(nxt);
  }
  if (lane == 0) {
    out5[0] = (float)mean;
    out5[1] = (float)sqrt(ss / (double)n);
    out5[2] = __uint_as_float(kmx); out5[3] = __uint_as_float(kmn);
    out5[4] = (n & 1) ? sel : (float)(((double)sel + (double)sel2) * 0.5);
  }
}

// The same statistics for the three feature sequences of one utterance with the values held in
// registers (NJ per lane): one copy of the code, no shared-memory re-reads in the bisection.
template <int NJ>
__device__ __noinline__ void tail_stats_regs(const float* fe, const float* fm, const unsigned short* zf, int n, float* out15) {
  const int lane = threadIdx.x & 31;
#pragma unroll 1
  for (int q = 0; q < 3; ++q) {
    const float* src = q == 0 ? fe : fm;
    // keys order like the values: float bit patterns for the non-negative energies / magnitudes, the integers
    // themselves for the crossing counts (a handful of significant bits: the bisection below then takes <= 10
    // rounds instead of walking the ~25 bits in which the float patterns of small integers differ)
    const bool ints = q == 2;
    auto val = [&](uint32_t k) { return ints ? (float)k : __uint_as_float(k); };
    uint32_t key[NJ];
    float ps = 0.f;
    uint32_t kmn = 0xffffffffu, kmx = 0u;
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
      const int i = lane + 32 * j;
      key[j] = 0xffffffffu;
      if (i < n) {
        key[j] = ints ? (uint32_t)zf[i] : __float_as_uint(src[i]);
        ps += val(key[j]); kmn = min(kmn, key[j]); kmx = max(kmx, key[j]);
      }
    }
    const float inv_n = 1.0f / (float)n;
    const float meanf = (float)warp_reduce((double)ps, OpAddD()) * inv_n;     // float32 result: float divide is enough
    kmx = __reduce_max_sync(0xffffffffu, kmx);
    kmn = __reduce_min_sync(0xffffffffu, kmn);
    float pss = 0.f;
#pragma unroll
    for (int j = 0; j < NJ; ++j) if (lane + 32 * j < n) { const float d = val(key[j]) - meanf; pss += d * d; }
    const double ss = warp_reduce((double)pss, OpAddD());
    const int rank = (n - 1) >> 1;
    uint32_t prefix = kmn;
    const uint32_t diff = kmn ^ kmx;
    if (diff) {
      int b = 31 - __clz(diff);
      prefix = kmn & ~((2u << b) - 1u);
      int cnt_lo = 0, cnt_bin = n;
      while (b >= 0 && cnt_bin > 1) {
        const uint32_t trial = prefix | (1u << b);
        int c = 0;
#pragma unroll
        for (int j = 0; j < NJ; ++j) c += (key[j] < trial);
        c = __reduce_add_sync(0xffffffffu, c);
        if (rank < c) cnt_bin = c - cnt_lo;
        else { prefix = trial; cnt_bin = cnt_lo + cnt_bin - c; cnt_lo = c; }
        --b;
      }
      if (b >= 0) {      // a single key is left in [prefix, prefix + 2^(b+1)): fetch it
        const uint32_t hi = prefix + ((2u << b) - 1u);
        uint32_t k = 0xffffffffu;
#pragma unroll
        for (int j = 0; j < NJ; ++j) if (key[j] >= prefix && key[j] <= hi) k = min(k, key[j]);
        prefix = __reduce_min_sync(0xffffffffu, k);
      }
    }
    const float sel = val(prefix);
    float sel2 = sel;
    if (!(n & 1)) {
      int le = 0;
      uint32_t nxt = 0xffffffffu;
#pragma unroll
      for (int j = 0; j < NJ; ++j) { if (key[j] <= prefix) ++le; else nxt = min(nxt, key[j]); }
      le = __reduce_add_sync(0xffffffffu, le);
      nxt = __reduce_min_sync(0xffffffffu, nxt);
      if (le < rank + 2 && nxt != 0xffffffffu) sel2 = val(nxt);
    }
    if (lane == 0) {
      float* o = out15 + 5 * q;
      o[0] = meanf;
      o[1] = sqrtf((float)ss * inv_n);
      o[2] = val(kmx); o[3] = val(kmn);
      o[4] = (n & 1) ? sel : 0.5f * sel + 0.5f * sel2;
    }
  }
}

}  // namespace

// ---------------------------------------------------------------------------------------
// kChain: frame 256 / shift 128 -- the tail warps run the sample-stationary chain for the windowed pass
// (each sample converted once, window coefficients in registers).
template <bool kChain>
__global__ void __launch_bounds__(kPipeThreads, 1) frontend_pipe_kernel(const PcmArgs a) {
  extern __shared__ __align__(128) unsigned char smem[];
  const int R = a.ring_slots, nrec = a.n_rec;
  const PipeLayout L = make_pipe_layout(R, a.cap_groups, a.cap_frames, a.fl, nrec);
  unsigned char* s_ring = smem + L.ring;
  unsigned long long* s_gsum = reinterpret_cast<unsigned long long*>(smem + L.gsum);   // [2][capG]
  uint32_t* s_bits = reinterpret_cast<uint32_t*>(smem + L.bits);
  uint32_t* s_meta = reinterpret_cast<uint32_t*>(smem + L.meta);   // per group: crossings inside it, its first / last two bits
  float* s_win = reinterpret_cast<float*>(smem + L.win);
  int2* s_desc = reinterpret_cast<int2*>(smem + L.desc);
  int4* s_part = reinterpret_cast<int4*>(smem + L.part);                                // [2][kStreamWarps]
  double* s_consts = reinterpret_cast<double*>(smem + L.consts);                        // [2][8]
  uint64_t* bar_full = reinterpret_cast<uint64_t*>(smem + L.bars);
  uint64_t* bar_empty = bar_full + R;
  unsigned long long* s_head = reinterpret_cast<unsigned long long*>(smem + L.head);   // [2][capG]

  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  // kChain fixes frame 256 / shift 128 at compile time: divisions, edge handling and the generic loops fold away
  const int fl = kChain ? 256 : a.fl, fs = kChain ? 128 : a.fs;
  const bool hann = (a.window == DSP_WIN_HANNING);
  // frames are sums of whole groups: the stream warps are done with the samples after pass B
  const bool edges = kChain ? false : (((fl % kGroup) | (fs % kGroup)) != 0 || fl > 16384);

#pragma unroll 1
  for (int j = tid; j < fl; j += kPipeThreads) s_win[j] = a.win_f32[j];
  if (tid == 0) {
    for (int i = 0; i < R; ++i) { mbar_init(&bar_full[i], 1); mbar_init(&bar_empty[i], edges ? kStreamWarps : 1); }
    mbar_fence_init();
  }
  __syncthreads();

  // =========================================================================================
  // CONTROL WARP: work distribution + TMA producer
  // =========================================================================================
  // The two register regimes never meet again: everything inside this branch ends in a return.
  if (wid >= kStreamWarps) {
  if constexpr (kSplitRegs) asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kTailRegs));
  if (wid == kPipeWarps - 1) {
    // Lane 0 schedules and issues the bulk copies.  Bulk copies need 16-byte aligned addresses on both sides (and the
    // tiled tensor-map form faults on an inner coordinate that is not a multiple of 16 bytes, tools/tma_probe.cu), so an
    // utterance that starts `shift` = 1..7 samples above a 16-byte boundary (packed CSR batches of odd lengths, ragged
    // data, sliced tensors) is fetched FROM that boundary: the ring holds the aligned stream, sample i of the utterance at
    // stream position i + shift, and the stream warps carry the offset through their group algebra (pass A / B / F) --
    // nothing is moved twice on chip.  The descriptor hands them (utterance, length | shift << 20).
    if (lane != 0) return;
    int slot = 0, lap = 0, useq = 0;
    unsigned int u_next = atomicAdd(a.work_counter, 1u);
    for (;;) {
      const long long u = (long long)u_next;
      const bool done = u >= a.n_utts;
      int n = 0, shift = 0;
      const unsigned char* gsrc = nullptr;
      if (!done) {
        u_next = atomicAdd(a.work_counter, 1u);       // one index ahead: its latency hides behind the copies
        const int64_t off = a.offsets[u];
        n = a.lengths ? a.lengths[u] : (int)(a.offsets[u + 1] - off);
        const int16_t* src = a.samples + off;
        shift = n > 0 ? (int)((reinterpret_cast<uintptr_t>(src) & 15) >> 1) : 0;     // samples above the 16-byte boundary
        gsrc = reinterpret_cast<const unsigned char*>(src) - 2 * shift;
      }
      s_desc[useq & (kDescRing - 1)] = make_int2(done ? -1 : (int)u, n | (shift << 20));
      const int np = n + shift;                       // samples of the aligned stream
      const int nchunks = np > 0 ? (np + kChunkSamples - 1) / kChunkSamples : 1;
      uint32_t dst32 = smem_u32(s_ring) + (uint32_t)slot * kChunkBytes, full32 = smem_u32(&bar_full[slot]), empty32 = smem_u32(&bar_empty[slot]);
      auto next_slot = [&]() {
        dst32 += kChunkBytes; full32 += 8; empty32 += 8;
        if (++slot == R) { slot = 0; ++lap; dst32 = smem_u32(s_ring); full32 = smem_u32(bar_full); empty32 = smem_u32(bar_empty); }
      };
      auto wait_empty = [&]() { if (lap > 0) mbar_wait(empty32, (uint32_t)((lap - 1) & 1)); };
      // full 4 KB chunks first (running shared / global addresses, no per-chunk arithmetic), then the last,
      // possibly partial one.  The arrivals and copies on raw addresses stay inline asm: through ptx.cuh helpers the
      // compiler schedules this kernel's later passes differently.
#pragma unroll 1
      for (int c = 0; c + 1 < nchunks; ++c) {
        wait_empty();
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(full32), "r"((uint32_t)kChunkBytes) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(dst32), "l"(gsrc), "r"((uint32_t)kChunkBytes), "r"(full32) : "memory");
        gsrc += kChunkBytes;
        next_slot();
      }
      {
        wait_empty();
        const int s0 = (nchunks - 1) * kChunkSamples;
        const int cnt = np > 0 ? np - s0 : 0;
        const uint32_t bytes = ((uint32_t)cnt * 2u) & ~15u;
        // tail of < 8 samples by plain loads; the release of the arrive below publishes them
        int16_t* dst = reinterpret_cast<int16_t*>(s_ring + (size_t)slot * kChunkBytes);
        const int16_t* gs = reinterpret_cast<const int16_t*>(gsrc);
        for (int i = (int)(bytes >> 1); i < cnt; ++i) dst[i] = gs[i];
        if (bytes) {
          asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(full32), "r"(bytes) : "memory");
          asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                       ::"r"(dst32), "l"(gsrc), "r"(bytes), "r"(full32) : "memory");
        } else {
          asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(full32) : "memory");
        }
        next_slot();
      }
      ++useq;
      if (done) break;
    }
    return;
  }

  // =========================================================================================
  // TAIL WARPS: one warp per utterance record
  // =========================================================================================
  // warp ids: stream first, then the tail warps, control last (the scheduler favours high ids: the latency-bound
  // tail warps get the issue slots they can use, the throughput-bound stream warps fill the rest)
  const int twid = wid - kStreamWarps;
  if (twid >= 0 && twid < kMaxTailWarps) {
    if (!kBatchMode && twid >= nrec) return;
    double* cand = reinterpret_cast<double*>(smem + L.scratch + (size_t)twid * 256);

    // Window coefficients of the hop-128 / length-256 chain.  The chain reads 16-byte ALIGNED vectors whatever the
    // utterance's address: with the trimmed segment starting m = 0..7 samples above a 16-byte boundary, a lane owns
    // segment samples 8*(lane&15) - m .. +8 of every hop block and its coefficients are the window shifted by m
    // (c = 0: first half of a frame, c = 1: the second; the m samples in front of a block's first frame get weight 0
    // there -- they are the LAST m samples of the frame two blocks back, added by a small correction pass).  One code
    // path and one LDG.128 per block for every alignment; the registers are loaded per utterance (tail_chain below).

    long long tp[5] = {0, 0, 0, 0, 0}, tprev = clock64();
    auto tick = [&](int i) { if (a.prof) { const long long t = clock64(); tp[i] += t - tprev; tprev = t; } };
    for (int it = 0;; ++it) {
      const int batch = kBatchMode ? (it & 1) : 0;
      // nb = records per batch = tail warps at work (7 unless the per-utterance records of a many-frame geometry leave
      // room for fewer: pipe_kernel_plan); the other tail warps only keep the batch barriers' head counts
      const int nb = kBatchMode ? (nrec >> 1) : nrec;
      unsigned char* rec = smem + L.rec + (size_t)(kBatchMode ? batch * nb + min(twid, nb - 1) : twid) * L.rec_bytes;
      int* r_int = reinterpret_cast<int*>(rec);
      double* r_dbl = reinterpret_cast<double*>(rec + 64);
      double* r_e = reinterpret_cast<double*>(rec + L.rec_e);
      const unsigned short* r_z = reinterpret_cast<const unsigned short*>(rec + L.rec_z);
      unsigned short* r_zf = reinterpret_cast<unsigned short*>(rec + L.rec_zf);
      float* s_fe = reinterpret_cast<float*>(rec + L.rec_fe);   // indexed by full-utterance frame number
      float* s_fm = reinterpret_cast<float*>(rec + L.rec_fm);
      if constexpr (kBatchMode) bar_sync(kBarBatchFull + batch, kBatchBarThreads);
      else bar_sync(kBarRecFull + twid, kRecBarThreads);
      int u = r_int[0];
      if constexpr (kBatchMode) {
        if (u == -2) break;                                   // the closing batch: every tail warp leaves
        if (twid >= nb) u = -1;                               // a tail warp without a record slot
        if (u < 0) { __syncwarp(); bar_arrive(kBarBatchEmpty + batch, kBatchBarThreads); continue; }   // padding of the last batch
      } else {
        if (u < 0) break;
      }
      tick(0);
      const int n = r_int[1], f1 = r_int[2], thr = r_int[4], kmn_s = r_int[5], kmx_s = r_int[6];
      const double phi_d = r_dbl[0], inv_m = r_dbl[1], mu = r_dbl[2];
      const float phi = (float)phi_d;
      const int16_t* x = a.samples + a.offsets[u];

      // =========================== endpoint decision ===================================
      int start = 0, end = n, flagged = 0;
      if (f1 > 0) {
        const double v = (double)(f1 - 1) * (90.0 / 100.0);
        const bool top = v >= (double)(f1 - 1);
        int rank = top ? f1 - 1 : (int)floor(v);
        // float projections of the energies (monotone); kept in registers for the usual sizes
        constexpr int kKeyRegs = key_regs<kChain>();
        const bool in_regs = f1 <= 32 * kKeyRegs;
        uint32_t key[kKeyRegs];
        uint32_t kmin = 0xffffffffu, kmax = 0u;
        if (in_regs) {
#pragma unroll
          for (int j = 0; j < kKeyRegs; ++j) {
            const int f = lane + 32 * j;
            key[j] = f < f1 ? __float_as_uint((float)r_e[f]) : 0xffffffffu;
            if (f < f1) { kmin = min(kmin, key[j]); kmax = max(kmax, key[j]); }
          }
        } else {
#pragma unroll 1
          for (int f = lane; f < f1; f += 32) { const uint32_t k = __float_as_uint((float)r_e[f]); kmin = min(kmin, k); kmax = max(kmax, k); }
        }
        kmin = __reduce_min_sync(0xffffffffu, kmin);
        kmax = __reduce_max_sync(0xffffffffu, kmax);
        auto count_below = [&](uint32_t trial) {
          int c = 0;
          if (in_regs) {
#pragma unroll
            for (int j = 0; j < kKeyRegs; ++j) c += (key[j] < trial);
          } else {
#pragma unroll 1
            for (int f = lane; f < f1; f += 32) c += (__float_as_uint((float)r_e[f]) < trial);
          }
          return (int)__reduce_add_sync(0xffffffffu, c);
        };
        // ---- 90th percentile: bisection until <= 32 frames share the bin, then float64 ranking
        uint32_t prefix = kmin;
        unsigned long long span = 1ull;
        int cnt_lo = 0, cnt_bin = f1;
        {
          const uint32_t diff = kmin ^ kmax;
          if (diff) {
            int b = 31 - __clz(diff);
            prefix = kmin & ~((2u << b) - 1u);
            while (b >= 0 && cnt_bin > 8) {
              const uint32_t trial = prefix | (1u << b);
              const int c = count_below(trial);
              if (rank < c) cnt_bin = c - cnt_lo;
              else { prefix = trial; cnt_bin = cnt_lo + cnt_bin - c; cnt_lo = c; }
              --b;
            }
            span = 1ull << (b + 1);
          }
        }
        bool unresolved = false;
        if (cnt_bin > 32) { unresolved = true; cnt_bin = 32; }    // > 32 frames share one float: replay in float64
        const int r1 = unresolved ? 0 : rank - cnt_lo;
        // gather the candidates of the bin (ballot compaction into the warp's scratch)
        {
          int base = 0;
          if (in_regs) {
#pragma unroll
            for (int j = 0; j < kKeyRegs; ++j) {
              const bool in = key[j] >= prefix && (unsigned long long)(key[j] - prefix) < span && key[j] != 0xffffffffu;
              const unsigned m = __ballot_sync(0xffffffffu, in);
              if (in) { const int s = base + __popc(m & ((1u << lane) - 1u)); if (s < 32) cand[s] = r_e[lane + 32 * j]; }
              base += __popc(m);
            }
          } else {
#pragma unroll 1
            for (int f0 = 0; f0 < f1; f0 += 32) {
              const int f = f0 + lane;
              bool in = false;
              double e = 0.0;
              if (f < f1) {
                e = r_e[f];
                const uint32_t k = __float_as_uint((float)e);
                in = k >= prefix && (unsigned long long)(k - prefix) < span;
              }
              const unsigned m = __ballot_sync(0xffffffffu, in);
              if (in) { const int s = base + __popc(m & ((1u << lane) - 1u)); if (s < 32) cand[s] = e; }
              base += __popc(m);
            }
          }
        }
        __syncwarp();
        const double mine = lane < cnt_bin ? cand[lane] : INFINITY;
        int below = 0;
#pragma unroll 1
        for (int j = 0; j < cnt_bin; ++j) {
          const double o = __shfl_sync(0xffffffffu, mine, j);
          below += (o < mine) || (o == mine && j < lane);
        }
        const unsigned m1 = __ballot_sync(0xffffffffu, lane < cnt_bin && below == r1);
        const unsigned m2 = __ballot_sync(0xffffffffu, lane < cnt_bin && below == r1 + 1);
        const double ka = __shfl_sync(0xffffffffu, mine, __ffs(m1) - 1);
        double kb = m2 ? __shfl_sync(0xffffffffu, mine, __ffs(m2) - 1) : ka;
        if (!m2 && !top) {               // rank + 1 lies above the candidate bin
          double nxt = INFINITY;
#pragma unroll 1
          for (int f = lane; f < f1; f += 32) {
            const double e = r_e[f];
            const uint32_t k = __float_as_uint((float)e);
            if (k >= prefix && (unsigned long long)(k - prefix) >= span) nxt = fmin(nxt, e);
          }
          nxt = warp_min_d(nxt);
          kb = nxt == INFINITY ? ka : nxt;
        }
        if (top) kb = ka;
        __syncwarp();

        // ---- noise floors and thresholds (audio_processing.py:188-217,239-247), every lane alike
        const int nf = min(5, f1 / 10);
        double noise_e, noise_z;
        if (nf > 0) {
          double ve[10], vz[10];
#pragma unroll 1
          for (int i = 0; i < 2 * nf; ++i) { const int f = i < nf ? i : f1 - 2 * nf + i; ve[i] = r_e[f]; vz[i] = (double)r_z[f]; }
          noise_e = noise_mean(ve, 2 * nf);
          noise_z = noise_mean(vz, 2 * nf);
        } else {
          noise_e = INFINITY; noise_z = INFINITY;
#pragma unroll 1
          for (int f = lane; f < f1; f += 32) { noise_e = fmin(noise_e, r_e[f]); noise_z = fmin(noise_z, (double)r_z[f]); }
          noise_e = warp_min_d(noise_e); noise_z = warp_min_d(noise_z);
        }
        const double speech = np_lerp(ka, kb, v - floor(v));
        const double t1 = speech * a.hr;
        const double t2 = noise_e + (speech - noise_e) * a.lr;
        const double t3 = noise_z * a.zr;
        // Slack on the thresholds (DESIGN.md "numerics"): 2^-40 relative, the rounding of the three-term
        // energy formula at its largest possible magnitude, and the reference's mean-rounding term
        // |mu| * sqrt(fl * E) / m at E_max (sqrt(y) <= (y + 1) / 2), each with a >= 4x margin.
        const double emx = (double)__uint_as_float(kmax) * 1.0000002;
        const double dmax = (double)max(kmx_s - thr, thr - kmn_s) + 1.0;
        const double amx = (double)fl * dmax * dmax;
        const double eps = 1.0 / 1099511627776.0;  // 2^-40
        const double smax = 8.881784197001252e-16 /* 2^-50 */ *
                            (fabs(mu) * 0.5 * ((double)fl * emx + 1.0) * inv_m + amx * inv_m * inv_m);
        const double tol1 = eps * fabs(t1) + fabs(a.hr) * smax + smax + eps * emx;
        const double tol2 = eps * (fabs(noise_e) + fabs(a.lr) * (fabs(speech) + fabs(noise_e))) +
                            (fabs(1.0 - a.lr) + fabs(a.lr)) * smax + smax + eps * emx;
        int n3 = f1, n4 = -1, flag = unresolved ? 1 : 0;
#pragma unroll 1
        for (int f = lane; f < f1; f += 32) {
          const double e = r_e[f];
          if (e > t1) { n3 = min(n3, f); n4 = max(n4, f); }
          if (fabs(e - t1) <= tol1 && !(e == 0.0 && t1 == 0.0)) flag = 1;
          if (fabs(e - t2) <= tol2 && !(e == 0.0 && t2 == 0.0)) flag = 1;
        }
        n3 = __reduce_min_sync(0xffffffffu, n3);
        n4 = __reduce_max_sync(0xffffffffu, n4);
        flagged = __any_sync(0xffffffffu, flag);
        if (n4 >= 0) {
          int n2 = 0, n5 = f1 - 1;
#pragma unroll 1
          for (int f = lane; f < f1; f += 32)
            if (r_e[f] <= t2) { if (f < n3) n2 = max(n2, f + 1); if (f > n4) n5 = min(n5, f - 1); }
          n2 = __reduce_max_sync(0xffffffffu, n2);
          n5 = __reduce_min_sync(0xffffffffu, n5);
          int n1 = 0, n6 = f1 - 1;
#pragma unroll 1
          for (int f = lane; f < f1; f += 32)
            if ((double)r_z[f] <= t3) { if (f < n2) n1 = max(n1, f + 1); if (f > n5) n6 = min(n6, f - 1); }
          n1 = __reduce_max_sync(0xffffffffu, n1);
          n6 = __reduce_min_sync(0xffffffffu, n6);
          start = n1 * fs;
          end = min(n6 * fs + fl, n);
        }
      }
      __syncwarp();     // the energy array is dead from here on: it becomes the feature buffers
      tick(1);

      // =========================== windowed frame features =============================
      const int seg = end - start;
      // The trimmed segment has usually left L2 since the stream warps read it (the batch hand-off puts ~10 utterances
      // per SM between the two uses): ask for all of it now, so that the chain below waits for DRAM once, not per block.
      {
        const char* pbase = reinterpret_cast<const char*>(x + start);
#pragma unroll 1
        for (int o = lane * 128; o < 2 * seg; o += 32 * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(pbase + o));
      }
      const int f2 = frame_count32(seg, fl, fs);
      const double sc_e = inv_m * inv_m, sc_m = inv_m;
      const int zbase = start / fs;        // start is a multiple of the hop: feature frame t is frame zbase + t
      int f2_chain = 0;      // frames [0, f2_chain) by the chain path, the rest generically
      if (kChain && (start & 127) == 0 && seg >= 256) f2_chain = min(f2, (seg - 256) / 128 + 1);
      if constexpr (kChain) {
        if (f2_chain > 0) {
          // 16 lanes per chain, 2 chains; a chain covers `per` consecutive frames = per + 1 hop blocks.
          // A sample becomes a float once: 0x4B000000 | (k ^ 0x8000) is 2^23 + 32768 + k, minus the integer
          // 2^23 + 32768 + thr (exact), minus phi (one rounding); then four multiply-adds (two frame
          // positions x energy / magnitude).  Block i is the second half of frame i-1 and the first of frame i.
          const int chain = lane >> 4, sub = lane & 15;
          const int per = (f2_chain + 1) >> 1;
          const int fa = chain * per;
          const int nfr = min(per, f2_chain - fa);           // frames of this chain (<= 0: idle)
          const int last = max(nfr, 0);                      // last hop block this chain may touch
          const bool hi8 = (sub & 8) != 0, writer = (sub & 7) == 0;
          // block i at ptr[16 * i]; an idle chain re-reads the first block of the segment and stores nothing
          const int mal = (int)((reinterpret_cast<uintptr_t>(x + start) & 15) >> 1);       // = the utterance's shift: start is a multiple of 128
          float cw[2][8], cw2[2][8];
#pragma unroll
          for (int c = 0; c < 2; ++c)
#pragma unroll
            for (int q8 = 0; q8 < 8; ++q8) {
              const int pos = c * 128 + 8 * sub + q8 - mal;
              const float w = s_win[max(pos, 0)];
              cw[c][q8] = pos >= 0 ? w : 0.f; cw2[c][q8] = pos >= 0 ? w * w : 0.f;
            }
          const int4* ptr = reinterpret_cast<const int4*>(x + start - mal + 8 * sub + (nfr > 0 ? fa : 0) * 128);
          const float c1f = -(8388608.f + 32768.f) - (float)thr;
          const float scale = hi8 ? (float)sc_m : (float)sc_e;
          float* dst = (hi8 ? s_fm : s_fe) + zbase + fa - 1;   // frame fa + i - 1 at dst[i]
          float* dummy = reinterpret_cast<float*>(cand);
#if DSP_CHAIN_PACKED
          // Packed fp32x2 arithmetic (sm_100 FFMA2 / FADD2 / FMUL2): the two samples of a 32-bit word travel as one
          // 64-bit register pair from the conversion on -- (x + c1f) - phi, d * d and the four multiply-adds of a word are
          // ONE instruction each instead of two.  Same FMA-pipe time, two thirds of the issue slots (12 instead of 17
          // per word), and issue slots are what this kernel runs out of.  Even and odd samples accumulate separately and
          // are added when a block's sums leave the lane.
          f32x2 cep = pk2(0.f, 0.f), cmp = pk2(0.f, 0.f);   // first-half partials of the previous block
          f32x2 cwp[2][4], cw2p[2][4];
#pragma unroll
          for (int c = 0; c < 2; ++c)
#pragma unroll
            for (int k = 0; k < 4; ++k) { cwp[c][k] = pk2(cw[c][2 * k], cw[c][2 * k + 1]); cw2p[c][k] = pk2(cw2[c][2 * k], cw2[c][2 * k + 1]); }
          const f32x2 c1f2 = pk2(c1f, c1f), nphi2 = pk2(-phi, -phi);
          auto step = [&](const int4& q, int i) {
            const uint32_t w[4] = {(uint32_t)q.x, (uint32_t)q.y, (uint32_t)q.z, (uint32_t)q.w};
            f32x2 e0 = pk2(0.f, 0.f), m0 = e0, e1 = cep, m1 = cmp;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const uint32_t ub = w[k] ^ 0x80008000u;
              const float xlo = __uint_as_float(__byte_perm(ub, 0x4b000000u, 0x7610));
              const float xhi = __uint_as_float(__byte_perm(ub, 0x4b000000u, 0x7632));
              const f32x2 d = add2(add2(pk2(xlo, xhi), c1f2), nphi2);
              const f32x2 qq = mul2(d, d);
              const f32x2 aa = d & 0x7fffffff7fffffffull;
              e0 = fma2(cw2p[0][k], qq, e0); m0 = fma2(cwp[0][k], aa, m0);
              e1 = fma2(cw2p[1][k], qq, e1); m1 = fma2(cwp[1][k], aa, m1);
            }
            cep = e0; cmp = m0;
            const float e1s = hsum2(e1), m1s = hsum2(m1);
            // transposed reduction of (e1, m1) over the chain's 16 lanes
            const float send = hi8 ? e1s : m1s, keep = hi8 ? m1s : e1s;
            float vv = keep + __shfl_xor_sync(0xffffffffu, send, 8);
            vv += __shfl_xor_sync(0xffffffffu, vv, 4);
            vv += __shfl_xor_sync(0xffffffffu, vv, 2);
            vv += __shfl_xor_sync(0xffffffffu, vv, 1);
            // one unconditional store (a branch here makes the compiler give up the straight-line schedule of the loop:
            // +50 % in this phase): lanes with nothing to write hit the warp's scratch word
            *((writer && i >= 1 && i <= nfr) ? dst + i : dummy) = vv * scale;
          };
#else
          float ce = 0.f, cm = 0.f;                          // first-half partials of the previous block
          auto step = [&](const int4& q, int i) {
            const uint32_t w[4] = {(uint32_t)q.x, (uint32_t)q.y, (uint32_t)q.z, (uint32_t)q.w};
            float e0 = 0.f, m0 = 0.f, e1 = ce, m1 = cm;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const uint32_t ub = w[k] ^ 0x80008000u;
              const float dlo = (__uint_as_float(__byte_perm(ub, 0x4b000000u, 0x7610)) + c1f) - phi;
              const float dhi = (__uint_as_float(__byte_perm(ub, 0x4b000000u, 0x7632)) + c1f) - phi;
              const float qlo = dlo * dlo, qhi = dhi * dhi;
              const float alo = fabsf(dlo), ahi = fabsf(dhi);
              e0 = fmaf(cw2[0][2 * k], qlo, e0); m0 = fmaf(cw[0][2 * k], alo, m0);
              e1 = fmaf(cw2[1][2 * k], qlo, e1); m1 = fmaf(cw[1][2 * k], alo, m1);
              e0 = fmaf(cw2[0][2 * k + 1], qhi, e0); m0 = fmaf(cw[0][2 * k + 1], ahi, m0);
              e1 = fmaf(cw2[1][2 * k + 1], qhi, e1); m1 = fmaf(cw[1][2 * k + 1], ahi, m1);
            }
            ce = e0; cm = m0;
            // transposed reduction of (e1, m1) over the chain's 16 lanes
            const float send = hi8 ? e1 : m1, keep = hi8 ? m1 : e1;
            float vv = keep + __shfl_xor_sync(0xffffffffu, send, 8);
            vv += __shfl_xor_sync(0xffffffffu, vv, 4);
            vv += __shfl_xor_sync(0xffffffffu, vv, 2);
            vv += __shfl_xor_sync(0xffffffffu, vv, 1);
            // one unconditional store (a branch here makes the compiler give up the straight-line schedule of the loop:
            // +50 % in this phase): lanes with nothing to write hit the warp's scratch word
            *((writer && i >= 1 && i <= nfr) ? dst + i : dummy) = vv * scale;
          };
#endif
          // kInFlight hop blocks in flight per lane (the tail warps run this phase together and wait on L2 / HBM together:
          // 4 -> 6 in flight is 3.65 -> 3.24 ms per 100k utterances; before the batch hand-off the larger loop body cost
          // more in instruction misses than it hid in latency); loads past the chain's last block re-read that block.
          // ld.global.cs: by the time a batch is processed the segment has usually left L2 (hit rate ~10 %) and this is
          // its last use -- streaming loads keep the dead lines from displacing the ring's traffic (-4 % DRAM reads)
#ifndef DSP_CHAIN_INFLIGHT
#define DSP_CHAIN_INFLIGHT 6
#endif
          constexpr int kInFlight = DSP_CHAIN_INFLIGHT;
          int4 q[kInFlight];
          auto load_block = [&](int bi) -> int4 { return __ldcs(ptr + 16 * bi); };
#pragma unroll
          for (int j = 0; j < kInFlight; ++j) q[j] = load_block(min(j, last));
#pragma unroll 1
          for (int i = 0; i <= per; i += kInFlight) {       // uniform trip count: the shuffles are warp-wide
#pragma unroll
            for (int j = 0; j < kInFlight; ++j) { step(q[j], i + j); q[j] = load_block(min(i + j + kInFlight, last)); }
          }
          if (mal) {
            // the last mal samples of every chained frame t: segment samples 128 (t + 2) - mal .. 128 (t + 2), window
            // positions 256 - mal .. 256 = the first mal samples of aligned block t + 2 (one lane per frame, two frames
            // in flight per lane; the chain has just pulled these lines through L2).  The vector of the very last block
            // may reach past the utterance: that one is read sample by sample.
            __syncwarp();
            const int16_t* xs = x + start - mal;
            const int vec_frames = min(f2_chain, (n - start + mal - 8) / 128 - 1);      // frames whose whole vector lies inside the utterance
            float wc[7];
#pragma unroll
            for (int j = 0; j < 7; ++j) wc[j] = j < mal ? s_win[256 - mal + j] : 0.f;
            auto corr = [&](const int4& q, int t) {
              const uint32_t w[4] = {(uint32_t)q.x, (uint32_t)q.y, (uint32_t)q.z, (uint32_t)q.w};
              float ce = 0.f, cm = 0.f;
#pragma unroll
              for (int j = 0; j < 7; ++j) {
                const int k = (j & 1) ? ((int)w[j >> 1] >> 16) : sext16(w[j >> 1]);
                const float wd = wc[j] * ((float)(k - thr) - phi);
                ce = fmaf(wd, wd, ce); cm += fabsf(wd);
              }
              s_fe[zbase + t] += ce * (float)sc_e;
              s_fm[zbase + t] += cm * (float)sc_m;
            };
#pragma unroll 1
            for (int t = lane; t < f2_chain; t += 64) {
              const int t2 = t + 32;
              const bool v1 = t < vec_frames, h2 = t2 < f2_chain, v2 = t2 < vec_frames;
              int4 q1 = make_int4(0, 0, 0, 0), q2 = q1;
              if (v1) q1 = __ldg(reinterpret_cast<const int4*>(xs + 128 * (t + 2)));
              if (v2) q2 = __ldg(reinterpret_cast<const int4*>(xs + 128 * (t2 + 2)));
              auto scalar = [&](int tt) {
                const int16_t* pp = xs + 128 * (tt + 2);
                uint32_t w[4] = {0, 0, 0, 0};
#pragma unroll
                for (int j = 0; j < 7; ++j) if (j < mal) w[j >> 1] |= (uint32_t)(unsigned short)__ldg(pp + j) << (16 * (j & 1));
                return make_int4((int)w[0], (int)w[1], (int)w[2], (int)w[3]);
              };
              if (!v1) q1 = scalar(t);
              if (h2 && !v2) q2 = scalar(t2);
              corr(q1, t);
              if (h2) corr(q2, t2);
            }
          }
        }
      }
      if (f2_chain < f2) {
        const int sub = lane & (kLanesPerFrame - 1);
        const int slot = lane / kLanesPerFrame;
        constexpr int kSlots = 32 / kLanesPerFrame;
        // Generic windowed pass: kLanesPerFrame lanes per frame.  Whatever the frame's address (odd hops, packed CSR
        // batches), a lane reads 16-byte ALIGNED vectors: the frame starts mm = 0..7 samples into its first vector, the
        // window is indexed per sample (scalar shared-memory loads at j = 8 v - mm + i), and the samples outside
        // [0, valid) -- in front of the frame in its first vector, behind it in the last -- get weight 0.
#pragma unroll 1
        for (int t0 = f2_chain; t0 < f2; t0 += kSlots) {
          const int t = t0 + slot;
          float e = 0.f, m = 0.f;
          if (t < f2) {
            const int p = start + t * fs;
            const int valid = min(fl, end - p);
            const int mm = (int)((reinterpret_cast<uintptr_t>(x + p) & 15) >> 1);
            const int4* xv = reinterpret_cast<const int4*>(x + p - mm);
            const float gc1f = -(8388608.f + 32768.f) - (float)thr;
            const f32x2 gc1 = pk2(gc1f, gc1f), gphi = pk2(-phi, -phi);
            f32x2 e2 = pk2(0.f, 0.f), m2 = e2;
            const int nv = (mm + valid + 7) >> 3;
            auto acc8 = [&](const int4& q, int v) {
              const uint32_t w[4] = {(uint32_t)q.x, (uint32_t)q.y, (uint32_t)q.z, (uint32_t)q.w};
              const int j0 = 8 * v - mm;
              float ww[8];
              if (j0 >= 0 && j0 + 8 <= valid) {
#pragma unroll
                for (int i = 0; i < 8; ++i) ww[i] = s_win[j0 + i];
              } else {
#pragma unroll
                for (int i = 0; i < 8; ++i) { const int j = j0 + i; const bool in = (unsigned)j < (unsigned)valid; const float wv = s_win[in ? j : 0]; ww[i] = in ? wv : 0.f; }
              }
              if constexpr (kChain) {
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                  const float dlo = (float)(sext16(w[k]) - thr) - phi;
                  const float dhi = (float)(((int)w[k] >> 16) - thr) - phi;
                  const float alo = ww[2 * k] * dlo, ahi = ww[2 * k + 1] * dhi;
                  e = fmaf(alo, alo, e); m += fabsf(alo);
                  e = fmaf(ahi, ahi, e); m += fabsf(ahi);
                }
              } else {
                // the general geometries spend a third of their instructions here: the two samples of a word travel as one
                // packed fp32x2 pair, converted like the chain's (0x4B000000 | (k ^ 0x8000) = 2^23 + 32768 + k, minus the
                // integer part exactly, minus phi in one rounding): 7 instead of 10.5 instructions per sample
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                  const uint32_t ub = w[k] ^ 0x80008000u;
                  const float xlo = __uint_as_float(__byte_perm(ub, 0x4b000000u, 0x7610));
                  const float xhi = __uint_as_float(__byte_perm(ub, 0x4b000000u, 0x7632));
                  const f32x2 d = add2(add2(pk2(xlo, xhi), gc1), gphi);
                  const f32x2 av = mul2(pk2(ww[2 * k], ww[2 * k + 1]), d);
                  e2 = fma2(av, av, e2);
                  m2 = add2(av & 0x7fffffff7fffffffull, m2);
                }
              }
            };
            // four 16-byte loads in flight per lane (the samples come from L2); the specialised 256 / 128 instantiation
            // comes here for the one or two zero-padded frames behind its chain only: one compact loop there, its
            // hot code has to stay inside the instruction cache
            int vq = sub;
#pragma unroll 1
            for (; !kChain && vq + 3 * kLanesPerFrame < nv; vq += 4 * kLanesPerFrame) {
              const int4 q0 = __ldg(xv + vq), q1 = __ldg(xv + vq + kLanesPerFrame);
              const int4 q2 = __ldg(xv + vq + 2 * kLanesPerFrame), q3 = __ldg(xv + vq + 3 * kLanesPerFrame);
              acc8(q0, vq); acc8(q1, vq + kLanesPerFrame); acc8(q2, vq + 2 * kLanesPerFrame); acc8(q3, vq + 3 * kLanesPerFrame);
            }
#pragma unroll 1
            for (; vq < nv; vq += kLanesPerFrame) { const int4 q = __ldg(xv + vq); acc8(q, vq); }
            if constexpr (!kChain) { e += hsum2(e2); m += hsum2(m2); }
          }
#pragma unroll
          for (int o = kLanesPerFrame / 2; o > 0; o >>= 1) {
            e += __shfl_xor_sync(0xffffffffu, e, o);
            m += __shfl_xor_sync(0xffffffffu, m, o);
          }
          if (t < f2 && sub == 0) { s_fe[zbase + t] = (float)((double)e * sc_e); s_fm[zbase + t] = (float)((double)m * sc_m); }
          // zero-padded frame whose crossing count the stream warps could not take from a bit string: count it
          // from the samples (sign of window * (x - mean), zero is negative, audio_processing.py:119-132)
          const bool need_zc = t < f2 && r_zf[zbase + t] == 0xffffu;
          if (__any_sync(0xffffffffu, need_zc)) {
            int zc = 0;
            if (need_zc) {
              const int p = start + t * fs;
              const int valid = min(fl, end - p);
              auto pos = [&](int j) { return j < valid && s_win[j] > 0.f && ((int)__ldg(x + p + j) - thr) >= 0; };
#pragma unroll 1
              for (int j = sub; j < min(valid, fl - 1); j += kLanesPerFrame) zc += (pos(j) != pos(j + 1));
            }
#pragma unroll
            for (int o = kLanesPerFrame / 2; o > 0; o >>= 1) zc += __shfl_xor_sync(0xffffffffu, zc, o);
            __syncwarp();
            if (need_zc && sub == 0) r_zf[zbase + t] = (unsigned short)zc;
          }
        }
      }
      __syncwarp();
      tick(2);

      // =========================== outputs + statistics ================================
      const int64_t fo = a.feat_offsets[u];
#pragma unroll 1
      for (int t = lane; t < f2; t += 32) {
        if (a.out.energy) a.out.energy[fo + t] = s_fe[zbase + t];
        if (a.out.magnitude) a.out.magnitude[fo + t] = s_fm[zbase + t];
        if (a.out.zcr) a.out.zcr[fo + t] = (float)r_zf[zbase + t];
      }
      if (a.out.stats && f2 > 0) {
        float* stats = a.out.stats + (int64_t)u * kStats;
        if (f2 <= 32 * 6) tail_stats_regs<6>(s_fe + zbase, s_fm + zbase, r_zf + zbase, f2, stats);
        else if (f2 <= 32 * key_regs<kChain>()) tail_stats_regs<key_regs<kChain>()>(s_fe + zbase, s_fm + zbase, r_zf + zbase, f2, stats);
        else {
          float st[5];
          warp_stats([&](int i) { return s_fe[zbase + i]; }, f2, st);
          if (lane == 0) for (int k = 0; k < 5; ++k) stats[k] = st[k];
          warp_stats([&](int i) { return s_fm[zbase + i]; }, f2, st);
          if (lane == 0) for (int k = 0; k < 5; ++k) stats[5 + k] = st[k];
          warp_stats([&](int i) { return (float)r_zf[zbase + i]; }, f2, st);
          if (lane == 0) for (int k = 0; k < 5; ++k) stats[10 + k] = st[k];
        }
      }
      if (lane == 0) {
        int status = DSP_UTT_OK;
        if (seg <= 0) status = DSP_UTT_EMPTY; else if (f2 == 0) status = DSP_UTT_NO_FRAMES;
        if (a.out.start) a.out.start[u] = start;
        if (a.out.end) a.out.end[u] = end;
        if (a.out.n_epd_frames) a.out.n_epd_frames[u] = f1;
        if (a.out.n_frames) a.out.n_frames[u] = f2;
        if (a.out.status) a.out.status[u] = status;
        if (flagged) { const int s = atomicAdd(a.flag_count, 1); a.flag_list[s] = u; }
      }
      __syncwarp();
      if constexpr (kBatchMode) bar_arrive(kBarBatchEmpty + batch, kBatchBarThreads);
      else bar_arrive(kBarRecEmpty + twid, kRecBarThreads);
      tick(3);
    }
    if (a.prof && twid == 0 && lane == 0) for (int i = 0; i < 4; ++i) atomicAdd((unsigned long long*)&a.prof[8 + i], (unsigned long long)tp[i]);
    return;
  }
  return;
  }   // wid >= kStreamWarps
  if constexpr (kSplitRegs) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kStreamRegs));

  // =========================================================================================
  // STREAM WARPS
  // =========================================================================================
  const int swid = wid, stid = tid;
  const int nbs = kBatchMode ? (nrec >> 1) : nrec;       // records per batch (pipe_kernel_plan)
  int useq = 0, cslot = 0, clap = 0, rec_id = 0, rec_lap = 0;
  long long sp[8] = {0, 0, 0, 0, 0, 0, 0, 0}, sprev = clock64();
  auto stick = [&](int i) { if (a.prof) { const long long t = clock64(); sp[i] += t - sprev; sprev = t; } };
  for (;;) {
    mbar_wait(&bar_full[cslot], (uint32_t)(clap & 1));
    stick(0);
    const int2 dsc = s_desc[useq & (kDescRing - 1)];
    const int u = dsc.x;
    if (u < 0) break;
    const int par = useq & 1;
    unsigned char* rec = smem + L.rec + (size_t)rec_id * L.rec_bytes;
    int* r_int = reinterpret_cast<int*>(rec);
    // record slot hand-off with the tail warps: per record, or (batch mode) per batch of kBatch records
    auto rec_acquire = [&]() {
      if constexpr (kBatchMode) { if (rec_lap > 0 && rec_id % nbs == 0) bar_sync(kBarBatchEmpty + rec_id / nbs, kBatchBarThreads); }
      else { if (rec_lap > 0) bar_sync(kBarRecEmpty + rec_id, kRecBarThreads); }
    };
    auto rec_publish = [&]() {
      if constexpr (kBatchMode) { if (rec_id % nbs == nbs - 1) bar_arrive(kBarBatchFull + rec_id / nbs, kBatchBarThreads); }
      else bar_arrive(kBarRecFull + rec_id, kRecBarThreads);
      if (++rec_id == nrec) { rec_id = 0; ++rec_lap; }
    };
    // The ring holds the 16-byte aligned stream around the utterance: sample i sits at stream position i + sh
    // (sh = 0..7, per utterance).  Groups, chunks and bit strings are indexed by STREAM position; a frame that starts at
    // sample p is the run of whole groups from p / 64 minus the first sh samples of its first group plus the first sh
    // samples of the group behind its last one -- the "head" sums / head bits every group records next to its totals.
    const int n = dsc.y & 0xfffff, sh = dsc.y >> 20;
    const int np = n + sh;
    const int nchunks = np > 0 ? (np + kChunkSamples - 1) / kChunkSamples : 1;
    const int ng = (np + kGroup - 1) / kGroup;
    unsigned long long* gsum = s_gsum + (size_t)par * a.cap_groups;
    unsigned long long* head = s_head + (size_t)par * a.cap_groups;
    auto chunk_ptr = [&](int c) -> const unsigned char* {
      int s = cslot + c; if (s >= R) s -= R;
      return s_ring + (size_t)s * kChunkBytes;
    };
    auto at_pos = [&](int i) -> int {       // sample at stream position i
      return (int)reinterpret_cast<const int16_t*>(chunk_ptr(i >> 11))[i & (kChunkSamples - 1)];
    };
    // head masks: word w of a group's first vector keeps its samples below sh
    uint32_t hmask[4];
#pragma unroll
    for (int w = 0; w < 4; ++w) hmask[w] = (2 * w + 1 < sh) ? 0xffffffffu : ((2 * w < sh) ? 0x0000ffffu : 0u);

    // =========================== pass A: group sums, min, max =========================
    int S = 0;
    uint32_t mn2 = 0x7fff7fffu, mx2 = 0x80008000u;
    int mn = 32767, mx = -32768;
#pragma unroll 1
    for (int c = swid; c < nchunks; c += kStreamWarps) {
      int s = cslot + c, lp = clap; if (s >= R) { s -= R; ++lp; }
      if (c) mbar_wait(&bar_full[s], (uint32_t)(lp & 1));
      const int g = kGroupsPerChunk * c + lane;
      const int base = g * kGroup;
      if (sh && g == 0 && n > 0) {
        // the sh samples in front of the utterance belong to its neighbour: overwrite them with copies of sample 0
        // (min / max unaffected, the sum corrected here, the head sums / bits of group 0 consistent with it)
        volatile int16_t* fp = reinterpret_cast<volatile int16_t*>(s_ring + (size_t)s * kChunkBytes);
        const int16_t k0 = fp[sh];
        for (int i = 0; i < sh; ++i) fp[i] = k0;
        S -= sh * (int)k0;
        fence_proxy_async();                              // the slot is refilled by a bulk copy later
      }
      asm volatile("" ::: "memory");
      if (base + kGroup <= np) {
        unsigned char* gp = s_ring + (size_t)s * kChunkBytes + lane * (2 * kGroup);
        if (sh) {
          // head of the group: sums over its first sh samples (one masked vector)
          const int4 q = *reinterpret_cast<const int4*>(gp);
          const uint32_t x0 = (uint32_t)q.x & hmask[0], x1 = (uint32_t)q.y & hmask[1], x2 = (uint32_t)q.z & hmask[2], x3 = (uint32_t)q.w & hmask[3];
          const uint32_t h0 = __byte_perm(x0, x1, 0x7531), l0 = __byte_perm(x0, x1, 0x6420);
          const uint32_t h1 = __byte_perm(x2, x3, 0x7531), l1 = __byte_perm(x2, x3, 0x6420);
          const int hhh = dp4a_ss((int)h1, (int)h1, dp4a_ss((int)h0, (int)h0, 0));
          const int hhl = dp4a_su((int)h1, l1, dp4a_su((int)h0, l0, 0));
          const uint32_t hll = dp4a_uu(l1, l1, dp4a_uu(l0, l0, 0u));
          const int hs1 = 256 * dp4a_ss((int)h1, 0x01010101, dp4a_ss((int)h0, 0x01010101, 0)) + (int)dp4a_uu(l1, 0x01010101u, dp4a_uu(l0, 0x01010101u, 0u));
          const long long hs2 = (long long)hhh * 65536 + (long long)hhl * 512 + (long long)hll;
          head[g] = ((unsigned long long)hs2 << 24) | (unsigned long long)((uint32_t)hs1 & 0xffffffu);
        }
        int hh = 0, hl = 0, sumh = 0;
        uint32_t ll = 0, sl = 0;
        // fully unrolled on purpose: a compact 2-unit loop (L0-resident, measured) made pass A 8 % faster and the
        // kernel no faster -- the phases share the SM's issue slots, see DESIGN.md
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int4 q = *reinterpret_cast<const int4*>(gp + 16 * ((j + lane) & 7));   // rotated: conflict-free
          const uint32_t h0 = __byte_perm((uint32_t)q.x, (uint32_t)q.y, 0x7531), l0 = __byte_perm((uint32_t)q.x, (uint32_t)q.y, 0x6420);
          const uint32_t h1 = __byte_perm((uint32_t)q.z, (uint32_t)q.w, 0x7531), l1 = __byte_perm((uint32_t)q.z, (uint32_t)q.w, 0x6420);
          hh = dp4a_ss((int)h0, (int)h0, hh); hh = dp4a_ss((int)h1, (int)h1, hh);
          hl = dp4a_su((int)h0, l0, hl);      hl = dp4a_su((int)h1, l1, hl);
          ll = dp4a_uu(l0, l0, ll);           ll = dp4a_uu(l1, l1, ll);
          sumh = dp4a_ss((int)h0, 0x01010101, sumh); sumh = dp4a_ss((int)h1, 0x01010101, sumh);
          sl = dp4a_uu(l0, 0x01010101u, sl);  sl = dp4a_uu(l1, 0x01010101u, sl);
          mn2 = __vimin3_s16x2(mn2, (uint32_t)q.x, (uint32_t)q.y); mn2 = __vimin3_s16x2(mn2, (uint32_t)q.z, (uint32_t)q.w);
          mx2 = __vimax3_s16x2(mx2, (uint32_t)q.x, (uint32_t)q.y); mx2 = __vimax3_s16x2(mx2, (uint32_t)q.z, (uint32_t)q.w);
        }
        const int s1 = 256 * sumh + (int)sl;
        const long long s2 = (long long)hh * 65536 + (long long)hl * 512 + (long long)ll;
        S += s1;
        gsum[g] = ((unsigned long long)s2 << 24) | (unsigned long long)((uint32_t)s1 & 0xffffffu);
      } else if (base < np) {
        // The partial last group (r = 1..63 valid samples): whole vectors like a full group, the ragged vector masked
        // for the sums and filled with copies of the group's first sample for min / max.  (One sample at a time this
        // lane walked up to 63 dependent shared-memory loads while seven warps waited at the barrier: the barrier's share
        // of pass A on ragged batches was 47 %.)
        const unsigned char* gp = s_ring + (size_t)s * kChunkBytes + lane * (2 * kGroup);
        const int r = np - base;
        const uint32_t kf2 = ((uint32_t)(unsigned short)reinterpret_cast<const int16_t*>(gp)[0]) * 0x00010001u;
        // word w of a vector keeps its samples below cnt (cnt = valid samples of that vector, 0..8)
        auto wmask = [](int w, int cnt) { return (2 * w + 1 < cnt) ? 0xffffffffu : ((2 * w < cnt) ? 0x0000ffffu : 0u); };
        int hh = 0, hl = 0, sumh = 0;
        uint32_t ll = 0, sl = 0;
        int h_hh = 0, h_hl = 0, h_sumh = 0;
        uint32_t h_ll = 0, h_sl = 0;
#pragma unroll 1
        for (int v = 0; 8 * v < r; ++v) {
          int4 q = *reinterpret_cast<const int4*>(gp + 16 * v);
          const int cnt = min(8, r - 8 * v);
          uint32_t xw[4] = {(uint32_t)q.x, (uint32_t)q.y, (uint32_t)q.z, (uint32_t)q.w};
#pragma unroll
          for (int w = 0; w < 4; ++w) {
            const uint32_t mk = wmask(w, cnt);
            const uint32_t mmw = (xw[w] & mk) | (kf2 & ~mk);           // min / max: invalid halves repeat a valid sample
            mn2 = __vimin3_s16x2(mn2, mmw, mmw); mx2 = __vimax3_s16x2(mx2, mmw, mmw);
            xw[w] &= mk;                                               // sums: invalid halves are zero
          }
          const uint32_t h0 = __byte_perm(xw[0], xw[1], 0x7531), l0 = __byte_perm(xw[0], xw[1], 0x6420);
          const uint32_t h1 = __byte_perm(xw[2], xw[3], 0x7531), l1 = __byte_perm(xw[2], xw[3], 0x6420);
          hh = dp4a_ss((int)h0, (int)h0, hh); hh = dp4a_ss((int)h1, (int)h1, hh);
          hl = dp4a_su((int)h0, l0, hl);      hl = dp4a_su((int)h1, l1, hl);
          ll = dp4a_uu(l0, l0, ll);           ll = dp4a_uu(l1, l1, ll);
          sumh = dp4a_ss((int)h0, 0x01010101, sumh); sumh = dp4a_ss((int)h1, 0x01010101, sumh);
          sl = dp4a_uu(l0, 0x01010101u, sl);  sl = dp4a_uu(l1, 0x01010101u, sl);
          if (v == 0 && sh) {
            // head of the group: its first min(sh, r) samples (all inside this vector)
            const int hc = min(sh, r);
            const uint32_t y0 = xw[0] & wmask(0, hc), y1 = xw[1] & wmask(1, hc), y2 = xw[2] & wmask(2, hc), y3 = xw[3] & wmask(3, hc);
            const uint32_t g0 = __byte_perm(y0, y1, 0x7531), m0 = __byte_perm(y0, y1, 0x6420);
            const uint32_t g1 = __byte_perm(y2, y3, 0x7531), m1 = __byte_perm(y2, y3, 0x6420);
            h_hh = dp4a_ss((int)g1, (int)g1, dp4a_ss((int)g0, (int)g0, 0));
            h_hl = dp4a_su((int)g1, m1, dp4a_su((int)g0, m0, 0));
            h_ll = dp4a_uu(m1, m1, dp4a_uu(m0, m0, 0u));
            h_sumh = dp4a_ss((int)g1, 0x01010101, dp4a_ss((int)g0, 0x01010101, 0));
            h_sl = dp4a_uu(m1, 0x01010101u, dp4a_uu(m0, 0x01010101u, 0u));
          }
        }
        const int s1 = 256 * sumh + (int)sl;
        const long long s2 = (long long)hh * 65536 + (long long)hl * 512 + (long long)ll;
        const int h1s = 256 * h_sumh + (int)h_sl;
        const long long h2s = (long long)h_hh * 65536 + (long long)h_hl * 512 + (long long)h_ll;
        S += s1;
        gsum[g] = ((unsigned long long)s2 << 24) | (unsigned long long)((uint32_t)s1 & 0xffffffu);
        head[g] = ((unsigned long long)h2s << 24) | (unsigned long long)((uint32_t)h1s & 0xffffffu);
      }
    }
    mn = min(mn, min(sext16(mn2), (int)mn2 >> 16));
    mx = max(mx, max(sext16(mx2), (int)mx2 >> 16));
    S = __reduce_add_sync(0xffffffffu, S);
    mn = __reduce_min_sync(0xffffffffu, mn);
    mx = __reduce_max_sync(0xffffffffu, mx);
    if (lane == 0) s_part[par * kStreamWarps + swid] = make_int4(S, mn, mx, 0);
    stick(1);
    bar_sync(kBarStream, kStreamThreads);
    stick(2);
    {
      const int4 pp = lane < kStreamWarps ? s_part[par * kStreamWarps + lane] : make_int4(0, 32767, -32768, 0);
      S = __reduce_add_sync(0xffffffffu, pp.x);
      mn = __reduce_min_sync(0xffffffffu, pp.y);
      mx = __reduce_max_sync(0xffffffffu, pp.z);
    }
    const int N = n > 0 ? n : 1;
    int thr;
    { int q = S / N; if ((S % N) != 0 && S < 0) --q; thr = q + 1; }                    // floor(S/N) + 1
    if (stid == kStreamThreads - 1) {
      // float64 constants of the utterance (needed from pass F on; published by the next barrier)
      const long long Rm = (long long)S - (long long)N * thr;                          // in [-N, 0)
      const long long M = max((long long)N * mx - S, (long long)S - (long long)N * mn);
      double* cst = s_consts + par * 8;
      cst[0] = (double)Rm / (double)N;
      cst[1] = (M > 0) ? (double)N / (double)M : 1.0;
      cst[2] = (double)S / (double)N;
    }

    // =========================== pass B: sign bits ====================================
    // When k - thr fits 16 bits for every sample (always, unless a full-scale signal sits on a large DC
    // offset) the subtraction runs on the packed word: w - (thr << 16) has the sign of the high sample,
    // w * 65536 - (thr << 16) that of the low one -- one instruction each, no unpacking.
    const bool narrow = (mx - thr <= 32766) && (thr - mn <= 32768) && thr >= -32766 && thr <= 32767;
    // fastest form (whole-group frames, narrow range): max(min(k - thr + 1, 1), 0) on both halves of a word in
    // ONE instruction (VIADDMNMX.S16x2.RELU) is the pair of "above the mean" bits; acc + acc + r appends
    // them to an even-sample and an odd-sample bit plane.  Only the per-group record (crossings inside the
    // group, its first / last two bits) is needed downstream, the bit string itself is never stored.
    const bool fastb = narrow && !edges;        // whole-group frames, narrow range: the bit string itself is never stored
    // group record of whole-group frames: crossings inside the group | samples 0,2,4,6,8 | samples 1,3,5,7 | sample 62 | sample 63
    auto group_meta = [](uint32_t E, uint32_t O) {
      const uint32_t x1 = E ^ O, x2 = (O ^ (E >> 1)) & 0x7fffffffu;
      return (uint32_t)(__popc(x1) + __popc(x2)) | ((E & 0x1fu) << kMetaE) | ((O & 0xfu) << kMetaO) | ((E >> 31) << kMetaP) | ((O >> 31) << kMetaL);
    };
    if (narrow) {
      // max(min(k - thr + 1, 1), 0) on both halves of a word in ONE instruction (VIADDMNMX.S16x2.RELU) is the pair of
      // "above the mean" bits; a shift-add drops them into an even-sample and an odd-sample bit plane.  Whole-group
      // frames keep only the per-group record; ragged-edge frames keep the planes themselves (bit-string helpers above).
      const uint32_t t2 = ((uint32_t)(1 - thr) & 0xffffu) * 0x00010001u;
#pragma unroll 1
      for (int c = swid; c < nchunks; c += kStreamWarps) {
        int s = cslot + c; if (s >= R) s -= R;
        const int g = kGroupsPerChunk * c + lane;
        if (g * kGroup + kGroup <= np) {
          const unsigned char* gp = s_ring + (size_t)s * kChunkBytes + lane * (2 * kGroup);
          const int rot = lane & 7;
          // r = the two bits of a word at positions 0 and 16; r << c drops them into bit c of both planes at once, so a
          // word costs one compare and one shift-add, with no doubling chain (word k of processing unit pp: bit 4 pp + k)
          uint32_t acc0 = 0, acc1 = 0;
#pragma unroll
          for (int pp = 0; pp < 4; ++pp) {
            const int4 qa = *reinterpret_cast<const int4*>(gp + 16 * ((pp + rot) & 7));
            const int4 qb = *reinterpret_cast<const int4*>(gp + 16 * ((pp + 4 + rot) & 7));
            acc0 += __viaddmin_s16x2_relu((uint32_t)qa.x, t2, 0x00010001u) << (4 * pp + 0);
            acc1 += __viaddmin_s16x2_relu((uint32_t)qb.x, t2, 0x00010001u) << (4 * pp + 0);
            acc0 += __viaddmin_s16x2_relu((uint32_t)qa.y, t2, 0x00010001u) << (4 * pp + 1);
            acc1 += __viaddmin_s16x2_relu((uint32_t)qb.y, t2, 0x00010001u) << (4 * pp + 1);
            acc0 += __viaddmin_s16x2_relu((uint32_t)qa.z, t2, 0x00010001u) << (4 * pp + 2);
            acc1 += __viaddmin_s16x2_relu((uint32_t)qb.z, t2, 0x00010001u) << (4 * pp + 2);
            acc0 += __viaddmin_s16x2_relu((uint32_t)qa.w, t2, 0x00010001u) << (4 * pp + 3);
            acc1 += __viaddmin_s16x2_relu((uint32_t)qb.w, t2, 0x00010001u) << (4 * pp + 3);
          }
          // planes in processing order -> undo the rotation: bit a of E / O is sample 2a / 2a+1 of the group
          const uint32_t ep = __byte_perm(acc0, acc1, 0x5410), op = __byte_perm(acc0, acc1, 0x7632);
          const uint32_t E = __funnelshift_l(ep, ep, 4 * rot), O = __funnelshift_l(op, op, 4 * rot);
          if (!edges) s_meta[g] = group_meta(E, O);
          else { s_bits[2 * g] = E; s_bits[2 * g + 1] = O; }
        } else if (edges && g * kGroup < np) {
          // partial last group, one sample at a time
          uint32_t E = 0, O = 0;
#pragma unroll 1
          for (int i = 0; i < kGroup && g * kGroup + i < np; ++i) {
            const uint32_t bit = (at_pos(g * kGroup + i) - thr >= 0);
            if (i & 1) O |= bit << (i >> 1); else E |= bit << (i >> 1);
          }
          s_bits[2 * g] = E; s_bits[2 * g + 1] = O;
        } else if (sh && g * kGroup < np) {
          // partial last group of a shifted stream: the last whole frame may end inside its head -- first 9 bits only
          uint32_t m = 0;
          for (int i = 0; i < 9 && g * kGroup + i < np; ++i)
            if (at_pos(g * kGroup + i) - thr >= 0) m |= 1u << ((i & 1) ? kMetaO + (i >> 1) : kMetaE + (i >> 1));
          s_meta[g] = m;
        }
        // whole-group frames: this was the chunk's last read -- hand the slot back now, not after the warp's other chunks
        // (the producer refills the ring in order, and the next utterance's last chunks are the ones pass A ends up
        // waiting for); ragged-edge frames read their edges from the ring in pass F and release there
        __syncwarp();
        if (!edges && lane == 0) mbar_arrive(&bar_empty[s]);
      }
      if (edges && stid < 4) s_bits[2 * ng + stid] = 0;
    } else {
    // wide range (a full-scale signal on a large DC offset: k - thr does not fit 16 bits): one subtraction per sample
#pragma unroll 1
    for (int c = swid; c < nchunks; c += kStreamWarps) {
      int s = cslot + c; if (s >= R) s -= R;
      const int g = kGroupsPerChunk * c + lane;
      const int base = g * kGroup;
      uint32_t E = 0, O = 0;
      if (base < np) {
#pragma unroll 1
        for (int i = 0; i < kGroup && base + i < np; ++i) {
          const uint32_t bit = (at_pos(base + i) - thr >= 0);
          if (i & 1) O |= bit << (i >> 1); else E |= bit << (i >> 1);
        }
        s_bits[2 * g] = E; s_bits[2 * g + 1] = O;
        if (!edges) s_meta[g] = group_meta(E, O);      // whole-group frames read the group records
      }
    }
    if (stid < 4) s_bits[2 * ng + stid] = 0;
    }
    // ring slots back to the producer: every warp for every slot when pass F still reads samples (frame
    // edges), else only the owner of a chunk, right after its own pass B
    auto release_slots = [&]() {
      __syncwarp();
      if (edges) { for (int c = lane; c < nchunks; c += 32) { int s = cslot + c; if (s >= R) s -= R; mbar_arrive(&bar_empty[s]); } }
      else if (lane == 0) { for (int c = swid; c < nchunks; c += kStreamWarps) { int s = cslot + c; if (s >= R) s -= R; mbar_arrive(&bar_empty[s]); } }
    };
    if (!edges && !fastb) release_slots();
    stick(3);
    bar_sync(kBarStream, kStreamThreads);
    stick(4);

    // =========================== pass F: EPD frames -> record =========================
    rec_acquire();
    stick(5);
    {
      const double phi_d = s_consts[par * 8 + 0], inv_m = s_consts[par * 8 + 1];
      double* r_e = reinterpret_cast<double*>(rec + L.rec_e);
      unsigned short* r_z = reinterpret_cast<unsigned short*>(rec + L.rec_z);
      unsigned short* r_zf = reinterpret_cast<unsigned short*>(rec + L.rec_zf);
      int f1 = 0;
      if (a.do_epd && n >= fl) f1 = (n - fl) / fs + 1;
      const int f2full = frame_count32(n, fl, fs);
      const int64_t eo = (a.out.epd_energy || a.out.epd_zcr) ? a.epd_offsets[u] : 0;
      const long long thr2 = (long long)thr * thr;
      const int nfull = n >= fl ? (n - fl) / fs + 1 : 0;        // frames without zero padding
      const int fmax = max(nfull, f2full);
      // shifted stream (sh = 1..7): head corrections of a whole-group frame.  Sign changes at pairs (i, i+1):
      // even i pairs are bits of E ^ O, odd i pairs bits of O ^ (E >> 1) (E / O = the even / odd samples of the record).
      // Leaving the frame in front: the sh pairs i < sh of its first group; entering behind: the pair across the last
      // group boundary and the sh - 1 pairs i < sh - 1 of the next group.
      const uint32_t mA1 = (1u << ((sh + 1) >> 1)) - 1u, mA2 = (1u << (sh >> 1)) - 1u;
      const uint32_t mB1 = mA2, mB2 = sh ? (1u << ((sh - 1) >> 1)) - 1u : 0u;
      auto head_changes = [](uint32_t m, uint32_t m1, uint32_t m2) {
        const uint32_t E = (m >> kMetaE) & 0x1fu, O = (m >> kMetaO) & 0xfu;
        return __popc((E ^ O) & m1) + __popc((O ^ (E >> 1)) & m2);
      };
      auto unpack1 = [](unsigned long long pk) { return ((int)((uint32_t)pk << 8)) >> 8; };
      // ragged-edge geometries have few, long frames (98 of 1,102 samples at the reference's default): TWO lanes per
      // frame there, each taking half of the whole groups and of the bit string and one of the frame's two ragged ends,
      // on ONE code path; a butterfly exchange per frame.  (Written for 2 / 4 / 8 lanes; 4 measured slower -- 1.47 against
      // 1.29 ms per 20k utterances at 1102 / 441: the per-frame float64 epilogue every lane runs then repeats twice.)
      const bool pair = !kChain && edges;
      constexpr int kMaxLaneShift = 1;
      int lshift = 0;                                     // log2(lanes per frame)
      if (pair) { lshift = 1; while (lshift < kMaxLaneShift && (nfull << (lshift + 1)) <= 2 * kStreamThreads) ++lshift; }
      const int lpf = 1 << lshift;
      const int fstep = kStreamThreads >> lshift;
#pragma unroll 1
      for (int f0 = 0; f0 < fmax; f0 += fstep) {
        const int f = f0 + (stid >> lshift);
        const int sub = stid & (lpf - 1);
        const int half = sub;                               // (lane 0 of a frame's group stores its results)
        const unsigned act = __ballot_sync(0xffffffffu, f < nfull);     // the lanes that reach the exchange below
        if (f >= fmax) continue;
        const int p = f * fs;
        int zc = 0;
        int hb0 = 0, hb1 = 0, hbp = 0, hbl = 0;     // sign bits of the frame's samples 0, 1, fl-2, fl-1
        if (f < nfull) {
          long long s1, s2;
          if (!edges) {
            // whole groups only: sum k, sum k^2, crossings from the per-group records
            const int g0 = p / kGroup, gpf = fl / kGroup;
            int k1 = 0; long long k2 = 0;
            uint32_t prev = 0, m_first = 0, m_last = 0;
#pragma unroll 2
            for (int j = 0; j < gpf; ++j) {
              const unsigned long long pk = gsum[g0 + j];
              const uint32_t m = s_meta[g0 + j];
              k2 += (long long)(pk >> 24);
              k1 += unpack1(pk);
              zc += (int)(m & 0x7fu) + (int)(((m >> kMetaE) ^ prev) & (j ? 1u : 0u));
              prev = m >> kMetaL;
              if (j == 0) m_first = m;
              m_last = m;
            }
            if (sh) {
              const unsigned long long ha = head[g0], hb = head[g0 + gpf];
              const uint32_t mb = s_meta[g0 + gpf];
              k1 += unpack1(hb) - unpack1(ha);
              k2 += (long long)(hb >> 24) - (long long)(ha >> 24);
              zc += (int)(((mb >> kMetaE) ^ (m_last >> kMetaL)) & 1u) + head_changes(mb, mB1, mB2) - head_changes(m_first, mA1, mA2);
              hb0 = (m_first >> meta_bit(sh)) & 1; hb1 = (m_first >> meta_bit(sh + 1)) & 1;
              hbl = (mb >> meta_bit(sh - 1)) & 1;
              hbp = sh >= 2 ? (mb >> meta_bit(sh - 2)) & 1 : (m_last >> kMetaL) & 1;
            } else {
              hb0 = (m_first >> kMetaE) & 1; hb1 = (m_first >> kMetaO) & 1; hbp = (m_last >> kMetaP) & 1; hbl = (m_last >> kMetaL) & 1;
            }
            s1 = (long long)(k1 - fl * thr);
            s2 = k2 - 2ll * thr * (long long)k1 + (long long)fl * thr2;
          } else {
            // sum k, sum k^2 over stream positions [ps, qs): whole groups from their records, the two ragged ends as
            // "head" sums -- the first r samples of a group, straight from the ring with the byte-plane dot products
            // of pass A on whole vectors and one masked vector (a frame edge costs <= 8 vector steps, not <= 63 samples)
            long long k1 = 0, k2 = 0;
            const int ps = p + sh, qs = ps + fl;
            const int ga = ps / kGroup, gb = qs / kGroup;
            const int gspan = gb - ga;
#pragma unroll 4
            for (int g = ga + ((gspan * sub) >> lshift); g < ga + ((gspan * (sub + 1)) >> lshift); ++g) {
              const unsigned long long pk = gsum[g];
              k2 += (long long)(pk >> 24);
              k1 += (long long)unpack1(pk);
            }
            auto head = [&](int g, int r, long long sign) {
              const unsigned char* gp = chunk_ptr(g >> 5) + (g & 31) * (2 * kGroup);
              int hh = 0, hl = 0, sumh = 0;
              uint32_t ll = 0, sl = 0;
              const int nv = r >> 3, rem = r & 7;
#pragma unroll 1
              for (int v = 0; v <= nv; ++v) {
                if (v == nv && rem == 0) break;
                int4 q = *reinterpret_cast<const int4*>(gp + 16 * v);
                if (v == nv) {          // the ragged vector: keep its first rem samples
                  const uint32_t m0 = rem >= 2 ? 0xffffffffu : 0x0000ffffu;
                  const uint32_t m1 = rem >= 4 ? 0xffffffffu : (rem == 3 ? 0x0000ffffu : 0u);
                  const uint32_t m2 = rem >= 6 ? 0xffffffffu : (rem == 5 ? 0x0000ffffu : 0u);
                  const uint32_t m3 = rem == 7 ? 0x0000ffffu : 0u;
                  q.x &= m0; q.y &= m1; q.z &= m2; q.w &= m3;
                }
                const uint32_t h0 = __byte_perm((uint32_t)q.x, (uint32_t)q.y, 0x7531), l0 = __byte_perm((uint32_t)q.x, (uint32_t)q.y, 0x6420);
                const uint32_t h1 = __byte_perm((uint32_t)q.z, (uint32_t)q.w, 0x7531), l1 = __byte_perm((uint32_t)q.z, (uint32_t)q.w, 0x6420);
                hh = dp4a_ss((int)h0, (int)h0, hh); hh = dp4a_ss((int)h1, (int)h1, hh);
                hl = dp4a_su((int)h0, l0, hl);      hl = dp4a_su((int)h1, l1, hl);
                ll = dp4a_uu(l0, l0, ll);           ll = dp4a_uu(l1, l1, ll);
                sumh = dp4a_ss((int)h0, 0x01010101, sumh); sumh = dp4a_ss((int)h1, 0x01010101, sumh);
                sl = dp4a_uu(l0, 0x01010101u, sl);  sl = dp4a_uu(l1, 0x01010101u, sl);
              }
              k1 += sign * (long long)(256 * sumh + (int)sl);
              k2 += sign * ((long long)hh * 65536 + (long long)hl * 512 + (long long)ll);
            };
            // (this branch always runs with lpf >= 2 lanes per frame; all of them execute the same instructions)
            {
              const bool first = sub == 0, lastl = sub == lpf - 1;
              if (first || lastl) {
                const int hr = (lastl ? qs : ps) & (kGroup - 1);
                if (hr) head(lastl ? gb : ga, hr, lastl ? 1 : -1);
              }
              // sign changes at the pairs (i, i + 1), i in [ps, qs - 1): lane j takes i in [b_j, b_(j+1))
              const int b0 = ps + (((qs - ps) * sub) >> lshift), b1 = ps + (((qs - ps) * (sub + 1)) >> lshift);
              zc = count_changes(s_bits, b0, lastl ? qs : b1 + 1);
#pragma unroll 1
              for (int o = 1; o < lpf; o <<= 1) {
                k1 += __shfl_xor_sync(act, k1, o); k2 += __shfl_xor_sync(act, k2, o); zc += __shfl_xor_sync(act, zc, o);
              }
            }
            s1 = k1 - (long long)fl * thr;
            s2 = k2 - 2ll * thr * k1 + (long long)fl * thr2;
            hb0 = bit_at(s_bits, ps); hb1 = bit_at(s_bits, ps + 1); hbl = bit_at(s_bits, qs - 1); hbp = bit_at(s_bits, qs - 2);
          }
          if (f < f1 && half == 0) {
            // exact integer sums of d = k - thr, then sum (d - phi)^2 in three roundings
            const double t1 = 2.0 * phi_d * (double)s1, t2 = (double)fl * phi_d * phi_d;
            const double ep = ((double)s2 - t1) + t2;
            const double e = ep * inv_m * inv_m;
            r_e[f] = e;
            r_z[f] = (unsigned short)zc;
            if (a.out.epd_energy) a.out.epd_energy[eo + f] = e;
            if (a.out.epd_zcr) a.out.epd_zcr[eo + f] = (float)zc;
          }
        }
        if (f < f2full && half == 0) {
          const int valid = min(fl, n - p);
          int zf;
          if (f < nfull && !(hann && fl <= 2)) {
            zf = zc;
            if (hann) zf += (hb1 - (hb0 ^ hb1)) + (hbp - (hbp ^ hbl));
          } else if (fastb) {
            zf = 0xffff;                     // zero-padded frame, no bit string in this mode: the tail counts it from L2
          } else {
            zf = frame_zcr(s_bits, p + sh, valid, fl, hann);
          }
          r_zf[f] = (unsigned short)zf;
        }
      }
      if (stid == kStreamThreads - 1) {
        r_int[0] = u; r_int[1] = n; r_int[2] = f1; r_int[3] = f2full; r_int[4] = thr; r_int[5] = mn; r_int[6] = mx;
        double* rd = reinterpret_cast<double*>(rec + 64);
        rd[0] = phi_d; rd[1] = inv_m; rd[2] = s_consts[par * 8 + 2];
      }
    }
    if (edges) release_slots();
    __syncwarp();
    rec_publish();
    cslot += nchunks; if (cslot >= R) { cslot -= R; ++clap; }
    ++useq;
    stick(6);
  }
  if (a.prof && stid == 0) { for (int i = 0; i < 7; ++i) atomicAdd((unsigned long long*)&a.prof[i], (unsigned long long)sp[i]); atomicAdd((unsigned long long*)&a.prof[15], (unsigned long long)useq); }
  if constexpr (kBatchMode) {
    // pad the open batch with "skip" records, then one closing batch that makes every tail warp leave
    auto mark = [&](int code) {
      if (rec_lap > 0 && rec_id % nbs == 0) bar_sync(kBarBatchEmpty + rec_id / nbs, kBatchBarThreads);
      if (stid == 0) *reinterpret_cast<int*>(smem + L.rec + (size_t)rec_id * L.rec_bytes) = code;
      __syncwarp();
      if (rec_id % nbs == nbs - 1) bar_arrive(kBarBatchFull + rec_id / nbs, kBatchBarThreads);
      if (++rec_id == nrec) { rec_id = 0; ++rec_lap; }
    };
#pragma unroll 1
    while (rec_id % nbs != 0) mark(-1);
#pragma unroll 1
    for (int k = 0; k < nbs; ++k) mark(-2);
    return;
  }
  // tell the tail warps to stop: one terminator record each
#pragma unroll 1
  for (int k = 0; k < nrec; ++k) {
    if (rec_lap > 0) bar_sync(kBarRecEmpty + rec_id, kRecBarThreads);
    if (stid == 0) *reinterpret_cast<int*>(smem + L.rec + (size_t)rec_id * L.rec_bytes) = -1;
    __syncwarp();
    bar_arrive(kBarRecFull + rec_id, kRecBarThreads);
    if (++rec_id == nrec) { rec_id = 0; ++rec_lap; }
  }
}

// ---------------------------------------------------------------------------------------
// Host side: capacity planning.  Returns false when the configuration does not fit this kernel
// (the caller falls back to frontend_pcm_kernel).
// ---------------------------------------------------------------------------------------
bool pipe_kernel_plan(int64_t max_len, int cap_frames, int fl, size_t smem_limit, PipePlan* plan) {
  if (max_len > 65535 || cap_frames > 65535 || fl > 65535) return false;      // 16-bit crossing counts, int32 sums
  const int chunks = (int)std::max<int64_t>((max_len + 7 + kChunkSamples - 1) / kChunkSamples, 1);   // + the <= 7 samples below a misaligned start
  const int capG = chunks * kGroupsPerChunk;
  if (kBatchMode) {
    // two batches of records, as many per batch (= tail warps at work) as leave the ring the utterance in flight plus
    // at least two chunks of the next one: 7 for the usual geometries, fewer when hops under ~100 samples make the
    // per-utterance records large (64/32 at 1 s: 1,377 frames, 16.6 KB per record -> 2 per batch)
    for (int nb = kBatch; nb >= 1; --nb) {
      const int nrec = 2 * nb;
      const PipeLayout fixed = make_pipe_layout(0, capG, cap_frames, fl, nrec);
      const long long room = (long long)smem_limit - fixed.total - 1024;
      int R = (int)(room / (kChunkBytes + 16));
      if (R > kMaxRingSlots) R = kMaxRingSlots;
      if (R < chunks + 2) continue;
      plan->ring_slots = R; plan->n_rec = nrec; plan->cap_groups = capG;
      plan->smem = (size_t)make_pipe_layout(R, capG, cap_frames, fl, nrec).total;
      return true;
    }
    return false;
  }
  for (int nrec = kMaxTailWarps; nrec >= 2; --nrec) {
    const PipeLayout fixed = make_pipe_layout(0, capG, cap_frames, fl, nrec);
    const long long room = (long long)smem_limit - fixed.total - 1024;        // static shared memory + slack
    int R = (int)(room / (kChunkBytes + 16));
    if (R > kMaxRingSlots) R = kMaxRingSlots;
    // two utterances in flight if possible; give up tail warps for ring slots otherwise
    const bool roomy = R >= 2 * chunks - 2 || R == kMaxRingSlots;
    if (R >= chunks + 1 && (roomy || nrec == 2)) {
      plan->ring_slots = R; plan->n_rec = nrec; plan->cap_groups = capG;
      plan->smem = (size_t)make_pipe_layout(R, capG, cap_frames, fl, nrec).total;
      return true;
    }
  }
  return false;
}

cudaError_t launch_frontend_pipe(const PcmArgs& a, int grid, size_t smem, cudaStream_t st) {
  const bool chain = (a.fl == 256 && a.fs == 128);
  auto fn = chain ? frontend_pipe_kernel<true> : frontend_pipe_kernel<false>;
  cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  fn<<<grid, kPipeThreads, smem, st>>>(a);
  return cudaGetLastError();
}

}  // namespace dsp
