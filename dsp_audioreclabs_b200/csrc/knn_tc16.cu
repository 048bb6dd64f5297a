// KNN candidate filter for the 15-dim statistical features on the 5th-generation tensor cores
// (src/models.py:33-35,56-58 -> KNeighborsClassifier(n_neighbors=3); BASELINE configs[2]: 10^6 queries x 10^5 train rows).
//
// D = 15 is thin, but it is exactly ONE K = 16 step of a kind::f16 MMA once |t|^2 rides along as the 16th feature:
//
//     a(q) = (-2 q_0, ..., -2 q_14, 1)      b(t) = (t_0, ..., t_14, |t|^2)      a . b = |t|^2 - 2 q.t = score(q, t)
//
// so the accumulator IS the score and the epilogue does nothing but compare.  Operands are split into two fp16 planes
// (hi = fp16(x), lo = fp16(x - hi): 22 significant bits) and a tile is three MMAs, hi.hi + hi.lo + lo.hi, into one fp32
// accumulator -- the same certified-filter contract as the fp32 scan it replaces (csrc/knn.cu): the kernel only has to
// return 8 candidates and the 8th-best computed score; knn_rerank_kernel recomputes the candidates in float64,
// certifies the top k against a bound on this kernel's evaluation error and sends a query to the exhaustive float64
// rescan otherwise.  Neighbours and labels never depend on the reduced-precision arithmetic.
//
// One persistent CTA per SM, 576 threads:
//   warp 0      TMA producer (cp.async.bulk, no tensor map: the pack kernels write tiles in the tensor core's canonical
//               K-major no-swizzle layout, so a tile is ONE contiguous 8 KB copy): the work unit's QB query blocks of
//               128 ({hi, lo} x QB, double-buffered across work units) and a ring of 128-row train tiles
//   warp 1      one thread issues tcgen05.mma.cta_group::1.kind::f16, M 128 x N 128 x K 16, 3 QB per train tile
//               (QB query blocks x 3 split passes) into an accumulator of 4 / QB stages that fills TMEM
//               (4 / QB stages x QB query blocks x 128 columns = 512); tcgen05.commit frees the ring slot and publishes
//               the stage
//   warps 2-17  epilogue, one query per thread (TMEM lane = query row), 4 / QB warps per (lane group, query block) on
//               32 QB columns of every tile each: tcgen05.ld 32 columns at a time; a 3-input min tree gives the minimum of
//               each 8 scores and of the 32; only when that beats some lane's C-th best score does the lane look at the
//               offending 8 columns one by one.
//               After the first few thousand train rows that happens for a few columns in a thousand: the epilogue
//               costs ~0.6 instructions per pair and the kernel is bound by the TMEM -> register path (4 B per pair).
// QB = 2 (256-query units): a train tile (8 KB) serves 256 queries, which halves the L2 -> SM operand traffic and the
// per-tile barrier round trips per pair against QB = 1 (the scan moves 25 GB from L2 for 10^11 pairs).  QB = 1
// (128-query units) is chosen for pruned calls with few units per SM (knn_prune_unit_queries): a unit visits only the
// tiles near all of its queries, and 128 queries close on the curve need fewer of them (DESIGN.md §7 item 4).
#include <cuda_fp16.h>

#include <algorithm>
#include <climits>
#include <cmath>
#include <cstring>
#include <numeric>

#include <cub/block/block_scan.cuh>
#include <cub/device/device_radix_sort.cuh>

#include "kernels.cuh"
#include "knn.cuh"
#include "ptx.cuh"

namespace dsp {

namespace {

constexpr int kRows = 128;                       // rows of one operand tile (queries per block, train rows per tile)
constexpr int kK = 16;                           // padded feature dimension = one MMA K step
constexpr int kPlaneBytes = kRows * kK * 2;      // one fp16 plane of a tile: 4 KB
constexpr int kTileBytes = 2 * kPlaneBytes;      // {hi, lo}: 8 KB
constexpr int kMaxUnitQ = 2 * kRows;            // queries per work unit: QB = 1 or 2 query blocks (query padding: 256)
constexpr int kTStages = 16;                     // 128 KB of train tiles in flight; with the query buffers and the candidate lists the CTA owns its SM (all of TMEM is allocated)
constexpr int kMaxAccStages = 4;                 // QB = 1: 4 stages of 128 columns; QB = 2: 2 stages of 2 x 128
constexpr int kEpiWarps = 16;
constexpr int kTcThreads = 32 * (2 + kEpiWarps);
constexpr int kTmemCols = 512;
constexpr int kEpiThreads = 32 * kEpiWarps;
constexpr int kListBytes = 2 * kKnnCand * kEpiThreads * 4;     // per-thread candidate lists: scores and indices, [entry][thread]
// query buffers, train ring, candidate lists + mbarriers and the TMEM address slot
constexpr size_t tc_smem(int qb) { return 2 * (size_t)qb * kTileBytes + (size_t)kTStages * kTileBytes + kListBytes + 1024; }
// canonical K-major no-swizzle layout: core matrix = 8 rows x 16 bytes (128 B contiguous); the two core matrices along
// K of one 8-row group are adjacent (LBO = 128 B); row groups follow every 256 B (SBO)
constexpr uint32_t kLBO = 128, kSBO = 256;
// instruction descriptor (kind::f16): D = F32 (bit 4), A = B = F16, both K-major, N >> 3 at bit 17, M >> 4 at bit 24
constexpr uint32_t kIdesc = (1u << 4) | ((uint32_t)(kRows >> 3) << 17) | ((uint32_t)(kRows >> 4) << 24);
static_assert(8 * (4 + 2 * kTStages + 2 * kMaxAccStages) + 8 <= 512, "barrier block of the shared-memory plan (unit slots at 512)");
constexpr float kPadNorm = 30000.f;              // |t|^2 of padding rows: above every real score (knn_tc16_max_norm)

__device__ __forceinline__ float min3f(float a, float b, float c) { return fminf(fminf(a, b), c); }
__device__ __forceinline__ float min8(const uint32_t* v) {
  const float a = min3f(__uint_as_float(v[0]), __uint_as_float(v[1]), __uint_as_float(v[2]));
  const float b = min3f(__uint_as_float(v[3]), __uint_as_float(v[4]), __uint_as_float(v[5]));
  return fminf(min3f(a, b, __uint_as_float(v[6])), __uint_as_float(v[7]));
}

// element (row r, feature c) of a packed plane
__device__ __forceinline__ int plane_offset(int r, int c) { return (r >> 3) * (int)kSBO + (c >> 3) * (int)kLBO + (r & 7) * 16 + (c & 7) * 2; }

// ---------------------------------------------------------------------------------------
// pack: one thread per (padded) row.  is_query: a = (-2 x, 1); else b = (x, |x|^2).  Packed row r holds source row
// gather[r] (gather optional); its norm goes to norms[gather[r]].
// flags[0] = max |x|^2 (float bits), flags[1] |= 1 when a row does not fit the filter's range
// ---------------------------------------------------------------------------------------
__global__ void knn_tc16_pack_kernel(const double* __restrict__ x, int64_t rows, int64_t rows_padded, int d, bool is_query,
                                     unsigned char* __restrict__ packed, float* __restrict__ norms, int* __restrict__ flags,
                                     float max_norm, const int* __restrict__ gather) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  bool bad = false;
  float nf = 0.f;
  if (r < rows_padded) {
    const int64_t src = (r < rows && gather) ? gather[r] : r;
    double v[kK];
    double ss = 0.0;
#pragma unroll
    for (int c = 0; c < kK - 1; ++c) {
      v[c] = (r < rows && c < d) ? x[src * d + c] : 0.0;
      ss += v[c] * v[c];
    }
    bad = r < rows && !(ss <= (double)max_norm);         // also catches NaN / inf
    nf = (float)ss;
    if (is_query) {
#pragma unroll
      for (int c = 0; c < kK - 1; ++c) v[c] *= -2.0;
      v[kK - 1] = 1.0;
    } else {
      v[kK - 1] = r < rows ? ss : (double)kPadNorm;
    }
    if (bad) {
#pragma unroll
      for (int c = 0; c < kK; ++c) v[c] = 0.0;
    }
    __align__(16) __half hi[kK];
    __align__(16) __half lo[kK];
#pragma unroll
    for (int c = 0; c < kK; ++c) {
      const __half h = __float2half_rn((float)v[c]);
      hi[c] = h;
      lo[c] = __float2half_rn((float)(v[c] - (double)__half2float(h)));
    }
    unsigned char* tile = packed + (size_t)(r / kRows) * kTileBytes;
    const int rr = (int)(r % kRows);
#pragma unroll
    for (int c8 = 0; c8 < 2; ++c8) {
      *reinterpret_cast<uint4*>(tile + plane_offset(rr, 8 * c8)) = *reinterpret_cast<const uint4*>(hi + 8 * c8);
      *reinterpret_cast<uint4*>(tile + kPlaneBytes + plane_offset(rr, 8 * c8)) = *reinterpret_cast<const uint4*>(lo + 8 * c8);
    }
    if (norms && r < rows) norms[src] = nf;
  }
  if (r >= rows) nf = 0.f;
  nf = warp_reduce(bad ? 0.f : nf, [](float a, float b) { return fmaxf(a, b); });
  bad = __any_sync(0xffffffffu, bad);
  if ((threadIdx.x & 31) == 0) {
    atomicMax(&flags[0], __float_as_int(nf));                   // non-negative floats order like ints
    if (bad) atomicOr(&flags[1], 1);
  }
}

// ---------------------------------------------------------------------------------------
// filter
// ---------------------------------------------------------------------------------------
// The slow path: ONE out-of-line copy per list length.  A thread's candidate list lives in shared memory
// ([entry][thread]: conflict-free), so the function takes nothing but scalars -- 8 scores, their first train row, the
// current threshold -- and the 16 call sites of the epilogue (4 groups of 8 in each of 4 chunks of a tile) are a few
// moves and a CALL each.  The insertion is branch-free and shallow: slot s becomes min(max(left neighbour, d), itself),
// every slot from the OLD values.  Returns the new threshold (the C-th best score).
template <int C>
__device__ __noinline__ float tc16_slow8(float v0, float v1, float v2, float v3, float v4, float v5, float v6, float v7, int idx0,
                                         float thr, float* __restrict__ l_cd, int* __restrict__ l_ci) {
  const float v[8] = {v0, v1, v2, v3, v4, v5, v6, v7};
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float d = v[j];
    if (d < thr) {
      float cd[C]; int ci[C]; bool p[C];
#pragma unroll
      for (int s = 0; s < C; ++s) { cd[s] = l_cd[s * kEpiThreads]; ci[s] = l_ci[s * kEpiThreads]; p[s] = d < cd[s]; }
#pragma unroll
      for (int s = C - 1; s > 0; --s) {
        l_ci[s * kEpiThreads] = p[s] ? (p[s - 1] ? ci[s - 1] : idx0 + j) : ci[s];
        l_cd[s * kEpiThreads] = fminf(fmaxf(cd[s - 1], d), cd[s]);
      }
      l_ci[0] = p[0] ? idx0 + j : ci[0];
      l_cd[0] = fminf(cd[0], d);
      thr = fminf(fmaxf(cd[C - 2], d), cd[C - 1]);
    }
  }
  return thr;
}

// kC: candidates kept per query (k + 2 for k <= 3, else 8): a shorter list is inserted into less often (C ln(n / C)
// insertions per query, each executed by the whole warp for the one or two lanes that need it) and costs less per
// insertion; the float64 certificate decides, per query, whether it was enough.
template <int kC, int kQB>
__global__ void __launch_bounds__(kTcThreads, 1)
knn_tc16_filter_kernel(const unsigned char* __restrict__ qpacked, const unsigned char* __restrict__ tpacked, int64_t m, int n,
                       int units, int t_tiles, const int* __restrict__ qflags, int* __restrict__ cand_idx,
                       float* __restrict__ cand_worst, const float* __restrict__ thr0, const Tc16Work w) {
  constexpr int kUnitQ = kQB * kRows, kQBufBytes = kQB * kTileBytes, kAccStages = 4 / kQB;
  constexpr int kWarpsPerBlock = 4 / kQB, kWarpCols = 32 * kQB;     // epilogue warps per (lane group, query block)
  extern __shared__ __align__(1024) unsigned char smem[];
  // (a query outside the filter's range was packed as the zero vector: it gets candidates like any other and the rerank
  //  kernel sends it to the exhaustive float64 scan -- qflags is informational)
  unsigned char* s_q = smem;                                // [2][kQB blocks][hi | lo]
  unsigned char* s_t = smem + 2 * kQBufBytes;               // [kTStages][hi | lo]
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + 2 * kQBufBytes + (size_t)kTStages * kTileBytes);
  uint64_t* q_full = bars;
  uint64_t* q_empty = q_full + 2;
  uint64_t* t_full = q_empty + 2;
  uint64_t* t_empty = t_full + kTStages;
  uint64_t* acc_full = t_empty + kTStages;
  uint64_t* acc_empty = acc_full + kAccStages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + kAccStages);
  // per query buffer: {unit, tiles it visits, offset of its tile list or -1 for every tile}; unit -1 ends the work.
  // Written by the producer before the buffer's q_full arrival; the buffer is refilled only after the MMA thread's commit
  // AND every epilogue warp's arrival on q_empty, so the epilogue reads the unit it is about to process
  int4* s_info = reinterpret_cast<int4*>(reinterpret_cast<unsigned char*>(bars) + 512);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // every wait is the suspended form: the producer and the MMA thread wait for hundreds of cycles at a time, and a
  // spinning try_wait loop took 28 % of all issued instructions away from the epilogue warps that share their schedulers

  if (tid == 0) {
    for (int i = 0; i < 2; ++i) { mbar_init(&q_full[i], 1); mbar_init(&q_empty[i], 1 + kEpiWarps); }
    for (int i = 0; i < kTStages; ++i) { mbar_init(&t_full[i], 1); mbar_init(&t_empty[i], 1); }
    for (int i = 0; i < kAccStages; ++i) { mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], kEpiWarps); }
    mbar_fence_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      int s = 0; uint32_t ph = 0;
      int qb = 0; uint32_t qph = 0;
      const bool lists = w.tiles && !(w.kept && *w.kept > w.kept_limit);
      for (int i = 0;; ++i) {
        mbar_wait(&q_empty[qb], qph ^ 1u);
        const int slot = w.counter ? atomicAdd(w.counter, 1) : (int)blockIdx.x + i * (int)gridDim.x;
        const int u = slot < units ? (w.unit_order ? w.unit_order[slot] : slot) : -1;
        const int cnt = (u >= 0 && lists) ? w.tile_count[u] : t_tiles, list = (u >= 0 && lists) ? u * w.stride : -1;
        s_info[qb] = make_int4(u, cnt, list, 0);
        if (u < 0) { mbar_arrive(&q_full[qb]); break; }
        mbar_expect_tx(&q_full[qb], (uint32_t)kQBufBytes);
        bulk_g2s(smem_u32(s_q + (size_t)qb * kQBufBytes), qpacked + (size_t)u * kQBufBytes, kQBufBytes, &q_full[qb]);
        if (++qb == 2) { qb = 0; qph ^= 1u; }
        int tb = cnt > 0 ? (list < 0 ? 0 : w.tiles[list]) : 0;
        for (int j = 0; j < cnt; ++j) {
          const int tb_next = j + 1 < cnt ? (list < 0 ? j + 1 : w.tiles[list + j + 1]) : 0;
          mbar_wait(&t_empty[s], ph ^ 1u);
          mbar_expect_tx(&t_full[s], (uint32_t)kTileBytes);
          bulk_g2s(smem_u32(s_t + (size_t)s * kTileBytes), tpacked + (size_t)tb * kTileBytes, kTileBytes, &t_full[s]);
          if (++s == kTStages) { s = 0; ph ^= 1u; }
          tb = tb_next;
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===== MMA issuer: one thread =====
    if (lane == 0) {
      int s = 0, as = 0, qb = 0; uint32_t ph = 0, aph = 0, qph = 0;
      for (;;) {
        mbar_wait(&q_full[qb], qph);
        tc_fence_after();
        const int4 info = s_info[qb];
        if (info.x < 0) break;
        const uint32_t q0 = smem_u32(s_q + (size_t)qb * kQBufBytes);
        for (int tb = 0; tb < info.y; ++tb) {
          mbar_wait(&acc_empty[as], aph ^ 1u);             // the epilogue has drained this accumulator stage
          mbar_wait(&t_full[s], ph);
          tc_fence_after();
          const uint32_t t_hi = smem_u32(s_t + (size_t)s * kTileBytes), t_lo = t_hi + kPlaneBytes;
#pragma unroll
          for (int h = 0; h < kQB; ++h) {
            const uint32_t q_hi = q0 + (uint32_t)h * kTileBytes, q_lo = q_hi + kPlaneBytes;
            const uint32_t d_tmem = tmem_base + (uint32_t)((as * kQB + h) * kRows);
            umma_f16(d_tmem, umma_desc<kLBO, kSBO>(q_hi), umma_desc<kLBO, kSBO>(t_hi), kIdesc, 0u);
            umma_f16(d_tmem, umma_desc<kLBO, kSBO>(q_hi), umma_desc<kLBO, kSBO>(t_lo), kIdesc, 1u);
            umma_f16(d_tmem, umma_desc<kLBO, kSBO>(q_lo), umma_desc<kLBO, kSBO>(t_hi), kIdesc, 1u);
          }
          umma_commit(&t_empty[s]);                         // ring slot free once these MMAs have read it
          umma_commit(&acc_full[as]);                       // every query block of this stage is complete
          if (++s == kTStages) { s = 0; ph ^= 1u; }
          if (++as == kAccStages) { as = 0; aph ^= 1u; }
        }
        umma_commit(&q_empty[qb]);                          // the unit's queries are no longer read
        if (++qb == 2) { qb = 0; qph ^= 1u; }
      }
    }
    __syncwarp();
  } else {
    // ===== epilogue: TMEM lane group = warp % 4 (hardware rule); (warp - 2) / 4 picks the query block and, with
    // kWarpsPerBlock warps per (lane group, query block), the kWarpCols columns of every tile the warp compares =====
    const int lg = warp & 3, grp = (warp - 2) >> 2;
    const int h = grp / kWarpsPerBlock, part = grp % kWarpsPerBlock;
    const int et = tid - 64;                                   // epilogue thread
    float* l_cd = reinterpret_cast<float*>(smem + 2 * kQBufBytes + (size_t)kTStages * kTileBytes + 1024) + et;     // behind the barrier block
    int* l_ci = reinterpret_cast<int*>(l_cd - et + kKnnCand * kEpiThreads) + et;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(lg * 32) << 16);
    int as = 0, qb = 0; uint32_t aph = 0, qph = 0;
    for (;;) {
      mbar_wait(&q_full[qb], qph);
      const int4 info = s_info[qb];
      __syncwarp();
      if (lane == 0) mbar_arrive(&q_empty[qb]);
      if (++qb == 2) { qb = 0; qph ^= 1u; }
      const int u = info.x, cnt = info.y, list = info.z;
      if (u < 0) break;
      auto tile_row = [&](int j) { return (list < 0 ? j : w.tiles[list + j]) * kRows; };      // packed position of the tile's row 0
#pragma unroll
      for (int c = 0; c < kKnnCand; ++c) { l_cd[c * kEpiThreads] = INFINITY; l_ci[c * kEpiThreads] = -1; }
      // thr0 (optional): the caller knows an upper bound on the query's k-th distance (row-sharded KNN: the k-th distance
      // within the shard that owns the query) -- the filter starts AT that threshold instead of paying ~C ln(n / C)
      // insertions per query to find its own, and never rises above it while its list is still filling
      const int64_t q_own = (int64_t)u * kUnitQ + h * kRows + lg * 32 + lane;
      const int64_t q_idx = q_own < m ? (w.qperm ? (int64_t)w.qperm[q_own] : q_own) : -1;
      const float thr_cap = (thr0 && q_idx >= 0) ? thr0[q_idx] : INFINITY;
      float thr = thr_cap;
      // Fast path: the minimum of each 8 scores and of all 32 by 3-input mins, all in registers.  A group of 8 whose
      // minimum beats the thread's C-th best goes to tc16_slow8.  History of this path (1 M x 100 k on one B200, the
      // TMEM -> register pipeline alone takes 7.9 ms): 128 unrolled register insertions (100+ KB of SASS, instruction-
      // cache misses on every excursion) 170 ms; reloading the offending 8 columns from TMEM 33 ms; selects + rolled loop,
      // bubble sort 31 ms; 5-entry list + min/max network 22 ms; out-of-line slow path + 64-column loads: DESIGN.md.
      auto process = [&](const uint32_t* v, int idx0) {
        const float s0 = min8(v), s1 = min8(v + 8), s2 = min8(v + 16), s3 = min8(v + 24);
        if (fminf(fminf(s0, s1), fminf(s2, s3)) < thr) {
#define DSP_TC16_GROUP(g, sg)                                                                                                     \
          if (sg < thr)                                                                                                          \
            thr = fminf(thr_cap, tc16_slow8<kC>(__uint_as_float(v[8 * g]), __uint_as_float(v[8 * g + 1]), __uint_as_float(v[8 * g + 2]), \
                                 __uint_as_float(v[8 * g + 3]), __uint_as_float(v[8 * g + 4]), __uint_as_float(v[8 * g + 5]),        \
                                 __uint_as_float(v[8 * g + 6]), __uint_as_float(v[8 * g + 7]), idx0 + 8 * g, thr, l_cd, l_ci));
          DSP_TC16_GROUP(0, s0) DSP_TC16_GROUP(1, s1) DSP_TC16_GROUP(2, s2) DSP_TC16_GROUP(3, s3)
#undef DSP_TC16_GROUP
        }
        __syncwarp();
      };
      // kWarpsPerBlock warps per (lane group, query block), each on its own kWarpCols columns of every tile with its own
      // candidate list: four epilogue warps per scheduler hide one another's TMEM-load and min-tree latencies (with two,
      // issue slots were 28 % busy and the tensor pipe 20 %), the accumulator stage goes back to the MMA thread as soon
      // as the warp's scores are in registers, and the lists are merged once per work unit.
      uint32_t va[32], vb[32];
      int row_next = cnt > 0 ? tile_row(0) : 0;
      for (int tb = 0; tb < cnt; ++tb) {
        const int base = row_next + part * kWarpCols;
        if (tb + 1 < cnt) row_next = tile_row(tb + 1);
        mbar_wait(&acc_full[as], aph);
        tc_fence_after();
        const uint32_t col = (uint32_t)((as * kQB + h) * kRows + part * kWarpCols);
        tmem_ld32(lane_addr + col, va);
        if constexpr (kQB == 2) tmem_ld32(lane_addr + col + 32, vb);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&acc_empty[as]);
        if (++as == kAccStages) { as = 0; aph ^= 1u; }
        process(va, base);
        if constexpr (kQB == 2) process(vb, base + 32);
      }
      // merge: the warp of part 0 folds the lists of its (lane group, query block)'s other warps (128, 256, 384 epilogue
      // threads up) into its own
      const int pair_bar = 1 + lg + 4 * h;
      bar_sync(pair_bar, 32 * kWarpsPerBlock);
      if (part == 0) {
        float cd[kC]; int ci[kC];
#pragma unroll
        for (int c = 0; c < kC; ++c) { cd[c] = l_cd[c * kEpiThreads]; ci[c] = l_ci[c * kEpiThreads]; }
#pragma unroll
        for (int p = 1; p < kWarpsPerBlock; ++p) {
#pragma unroll
          for (int b = 0; b < kC; ++b) {
            float d = l_cd[b * kEpiThreads + p * 128]; int i = l_ci[b * kEpiThreads + p * 128];
#pragma unroll
            for (int c = 0; c < kC; ++c) {          // sorted insertion: carry the displaced entry down the list
              if (d < cd[c]) { const float td = cd[c]; const int ti = ci[c]; cd[c] = d; ci[c] = i; d = td; i = ti; }
            }
          }
        }
#pragma unroll
        for (int c = 0; c < kC; ++c) { l_cd[c * kEpiThreads] = cd[c]; l_ci[c * kEpiThreads] = ci[c]; }
      }
      if (part == 0 && q_idx >= 0) {
#pragma unroll
        for (int c = 0; c < kKnnCand; ++c) {
          const int i = c < kC ? l_ci[c * kEpiThreads] : -1;
          cand_idx[q_idx * kKnnCand + c] = (i < 0 || !w.tperm) ? i : (i < n ? w.tperm[i] : -1);      // padding rows: none
        }
        cand_worst[q_idx] = l_cd[(kC - 1) * kEpiThreads];
      }
      // the other warps must not re-initialise their lists for the next unit before they have been read
      bar_sync(pair_bar, 32 * kWarpsPerBlock);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}


// ---------------------------------------------------------------------------------------
// tile pruning (knn.cuh): everything here runs once per call before the main filter pass, block = one work unit
// ---------------------------------------------------------------------------------------
// Every kernel here is built for both unit sizes: kPruneThreads = queries per unit, one thread per query.
// Skip test: LB(unit box, tile box) > U (1 + kPruneRel).  The margin covers the eigenvectors' deviation from exact
// orthonormality (|V^T V - I| ~ 1e-14 after Jacobi) and the float64 rounding of the distances; the rounding of the
// projections is covered by the per-box slack, which is subtracted from every axis gap.
constexpr double kPruneRel = 1e-9;
// per box: projection error <= 16 eps |x - mean|_1 (15 products, sequential sums); 1e-13 |x - mean|_1 bounds it 60x over
constexpr double kPruneSlack = 1e-13;

__device__ __forceinline__ double prune_project(const double* __restrict__ x, const KnnPruneGeom* __restrict__ g, int d, int na,
                                                double* __restrict__ p) {
  double c[kPruneMaxDim];
  double l1 = 0.0;
#pragma unroll
  for (int j = 0; j < kPruneMaxDim; ++j) { c[j] = j < d ? x[j] - g->mean[j] : 0.0; l1 += fabs(c[j]); }
#pragma unroll
  for (int a = 0; a < kPruneMaxDim; ++a) {
    if (a >= na) break;
    double s = 0.0;
    for (int j = 0; j < d; ++j) s += c[j] * g->axis[a][j];
    p[a] = s;
  }
  return l1;
}

// key of the query order: Morton code of the first three projections, 10 bits each over the train set's range
__global__ void knn_prune_keys_kernel(const double* __restrict__ q, int64_t m, const KnnPruneGeom* __restrict__ g,
                                      unsigned* __restrict__ keys, int* __restrict__ vals) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= m) return;
  const int d = g->d, na = d < 3 ? d : 3;
  double p[kPruneMaxDim];
  prune_project(q + i * d, g, d, na, p);
  unsigned code = 0;
  for (int a = 0; a < na; ++a) {
    const double t = (p[a] - g->key_lo[a]) * g->key_scale[a];
    const unsigned v = t >= 0.0 ? (t < 1023.0 ? (unsigned)t : 1023u) : 0u;      // NaN -> 0
#pragma unroll
    for (int b = 0; b < 10; ++b) code |= ((v >> b) & 1u) << (3 * b + 2 - a);
  }
  keys[i] = code;
  vals[i] = (int)i;
}

template <int kPruneThreads>
__device__ __forceinline__ double block_max(double v, double* sh) {
  v = warp_reduce(v, [](double a, double b) { return fmax(a, b); });
  __syncthreads();
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
  __syncthreads();
  double r = sh[0];
  for (int w = 1; w < kPruneThreads / 32; ++w) r = fmax(r, sh[w]);
  return r;
}

// box of a unit's queries in the principal axes; queries outside the filter's range (rescanned in float64 anyway) and
// padding positions do not count
template <int kPruneThreads>
__global__ void __launch_bounds__(kPruneThreads)
knn_prune_unit_box_kernel(const double* __restrict__ q, int64_t m, const KnnPruneGeom* __restrict__ g, const int* __restrict__ qperm,
                          const float* __restrict__ qnorm, float qnorm_limit, double* __restrict__ ulo, double* __restrict__ uhi,
                          double* __restrict__ uslack) {
  __shared__ double s_lo[kPruneThreads / 32][kPruneMaxDim], s_hi[kPruneThreads / 32][kPruneMaxDim], s_red[kPruneThreads / 32];
  const int u = blockIdx.x, d = g->d, w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t pos = (int64_t)u * kPruneThreads + threadIdx.x;
  const int64_t qi = pos < m ? qperm[pos] : -1;
  const bool valid = qi >= 0 && qnorm[qi] <= qnorm_limit;
  double p[kPruneMaxDim], l1 = 0.0;
  if (valid) l1 = prune_project(q + qi * d, g, d, d, p);
#pragma unroll
  for (int a = 0; a < kPruneMaxDim; ++a) {
    if (a >= d) break;
    const double lo = warp_reduce(valid ? p[a] : INFINITY, [](double x, double y) { return fmin(x, y); });
    const double hi = warp_reduce(valid ? p[a] : -INFINITY, [](double x, double y) { return fmax(x, y); });
    if (lane == 0) { s_lo[w][a] = lo; s_hi[w][a] = hi; }
  }
  const double l1max = block_max<kPruneThreads>(l1, s_red);            // (its barriers also publish s_lo / s_hi)
  if (threadIdx.x < d) {
    double lo = INFINITY, hi = -INFINITY;
    for (int ww = 0; ww < kPruneThreads / 32; ++ww) { lo = fmin(lo, s_lo[ww][threadIdx.x]); hi = fmax(hi, s_hi[ww][threadIdx.x]); }
    ulo[(int64_t)u * d + threadIdx.x] = lo;
    uhi[(int64_t)u * d + threadIdx.x] = hi;
  }
  if (threadIdx.x == 0) uslack[u] = kPruneSlack * (1.0 + l1max);
}

__device__ __forceinline__ bool less_dt(double da, int ta, double db, int tb) { return da < db || (da == db && ta < tb); }

// seed lists: the kPruneSeedTiles tiles whose box centre is nearest the unit's box centre
template <int kPruneThreads>
__global__ void __launch_bounds__(kPruneThreads)
knn_prune_seed_kernel(int t_tiles, int d, const double* __restrict__ ulo, const double* __restrict__ uhi, const double* __restrict__ tlo,
                      const double* __restrict__ thi, int S, int* __restrict__ seed, int* __restrict__ seed_cnt) {
  __shared__ double s_d[kPruneThreads / 32];
  __shared__ int s_t[kPruneThreads / 32];
  __shared__ int s_win;
  const int u = blockIdx.x, w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  double c[kPruneMaxDim];
  for (int a = 0; a < d; ++a) c[a] = 0.5 * (ulo[(int64_t)u * d + a] + uhi[(int64_t)u * d + a]);
  double bd[kPruneSeedTiles];
  int bt[kPruneSeedTiles];
#pragma unroll
  for (int s = 0; s < kPruneSeedTiles; ++s) { bd[s] = INFINITY; bt[s] = INT_MAX; }
  for (int t = threadIdx.x; t < t_tiles; t += kPruneThreads) {
    double dd = 0.0;
    for (int a = 0; a < d; ++a) { const double x = c[a] - 0.5 * (tlo[(int64_t)t * d + a] + thi[(int64_t)t * d + a]); dd += x * x; }
    if (!(dd < INFINITY)) dd = INFINITY;               // a unit without queries in range: any tiles will do
    int s = kPruneSeedTiles - 1;
    if (!less_dt(dd, t, bd[s], bt[s])) continue;
    while (s > 0 && less_dt(dd, t, bd[s - 1], bt[s - 1])) { bd[s] = bd[s - 1]; bt[s] = bt[s - 1]; --s; }
    bd[s] = dd; bt[s] = t;
  }
  for (int r = 0; r < S; ++r) {
    double md = bd[0];
    int mt = bt[0];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double od = __shfl_xor_sync(0xffffffffu, md, o);
      const int ot = __shfl_xor_sync(0xffffffffu, mt, o);
      if (less_dt(od, ot, md, mt)) { md = od; mt = ot; }
    }
    if (lane == 0) { s_d[w] = md; s_t[w] = mt; }
    __syncthreads();
    if (threadIdx.x == 0) {
      for (int ww = 1; ww < kPruneThreads / 32; ++ww) if (less_dt(s_d[ww], s_t[ww], md, mt)) { md = s_d[ww]; mt = s_t[ww]; }
      s_win = mt;
      seed[(int64_t)u * S + r] = mt;
    }
    __syncthreads();
    if (bt[0] == s_win) {                               // tiles are distinct: one owner pops its head
#pragma unroll
      for (int s = 0; s + 1 < kPruneSeedTiles; ++s) { bd[s] = bd[s + 1]; bt[s] = bt[s + 1]; }
      bd[kPruneSeedTiles - 1] = INFINITY; bt[kPruneSeedTiles - 1] = INT_MAX;
    }
  }
  if (threadIdx.x == 0) seed_cnt[u] = S;
}

// U per query: the k-th float64 distance among the seed pass's candidates (real rows, so an upper bound on the k-th
// neighbour's distance), capped by the caller's bound; the unit's radius is the largest U of its queries in range
template <int kPruneThreads>
__global__ void __launch_bounds__(kPruneThreads)
knn_prune_bound_kernel(const double* __restrict__ train, const double* __restrict__ q, int64_t m, int d, int k,
                       const int* __restrict__ qperm, const int* __restrict__ cand_idx, const float* __restrict__ qnorm, float qnorm_limit,
                       const double* __restrict__ caller_bound, double* __restrict__ bound, double* __restrict__ unit_rad) {
  __shared__ double s_red[kPruneThreads / 32];
  const int u = blockIdx.x;
  const int64_t pos = (int64_t)u * kPruneThreads + threadIdx.x;
  const int64_t qi = pos < m ? qperm[pos] : -1;
  const bool valid = qi >= 0 && qnorm[qi] <= qnorm_limit;
  double U = INFINITY;
  if (qi >= 0) {
    double best[kKnnCand];
    int nb = 0;
    for (int c = 0; c < kKnnCand; ++c) {
      const int i = cand_idx[qi * kKnnCand + c];
      if (i < 0) continue;
      double dd = 0.0;                                   // sum_j (q_j - t_j)^2 in feature order, as knn_rerank computes it
      for (int j = 0; j < d; ++j) { const double x = q[qi * d + j] - train[(int64_t)i * d + j]; dd += x * x; }
      int s = nb++;
      while (s > 0 && dd < best[s - 1]) { best[s] = best[s - 1]; --s; }
      best[s] = dd;
    }
    if (nb >= k) U = best[k - 1];
    if (caller_bound) U = fmin(U, caller_bound[qi]);
    bound[qi] = U;
  }
  const double any = block_max<kPruneThreads>(valid ? 1.0 : 0.0, s_red);
  const double r = block_max<kPruneThreads>(valid ? U : -INFINITY, s_red);
  if (threadIdx.x == 0) unit_rad[u] = any > 0.0 ? r : INFINITY;      // no query in range: keep every tile
}

// the main pass's tile list of a unit, in tile order: every tile whose box may hold a row within the unit's radius
template <int kPruneThreads>
__global__ void __launch_bounds__(kPruneThreads)
knn_prune_list_kernel(int t_tiles, int d, const double* __restrict__ ulo, const double* __restrict__ uhi, const double* __restrict__ uslack,
                      const double* __restrict__ unit_rad, const double* __restrict__ tlo, const double* __restrict__ thi,
                      const double* __restrict__ tslack, int* __restrict__ tiles, int* __restrict__ count, int* __restrict__ unit_ids,
                      unsigned long long* __restrict__ kept) {
  using Scan = cub::BlockScan<int, kPruneThreads>;
  __shared__ typename Scan::TempStorage scan_tmp;
  __shared__ double s_lo[kPruneMaxDim], s_hi[kPruneMaxDim];
  const int u = blockIdx.x;
  if (threadIdx.x < d) { s_lo[threadIdx.x] = ulo[(int64_t)u * d + threadIdx.x]; s_hi[threadIdx.x] = uhi[(int64_t)u * d + threadIdx.x]; }
  __syncthreads();
  const double lim = unit_rad[u] * (1.0 + kPruneRel), sl_u = uslack[u];
  int run = 0;
  for (int base = 0; base < t_tiles; base += kPruneThreads) {
    const int t = base + threadIdx.x;
    int keep = 0;
    if (t < t_tiles) {
      const double sl = sl_u + tslack[t];
      double lb = 0.0;
      for (int a = 0; a < d; ++a) {
        const double gap = fmax(tlo[(int64_t)t * d + a] - s_hi[a], s_lo[a] - thi[(int64_t)t * d + a]) - sl;
        if (gap > 0.0) lb += gap * gap;
      }
      keep = lb <= lim;
    }
    int at, total;
    Scan(scan_tmp).ExclusiveSum(keep, at, total);
    if (keep) tiles[(int64_t)u * t_tiles + run + at] = t;
    run += total;
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    count[u] = run;
    unit_ids[u] = u;
    atomicAdd(kept, (unsigned long long)run);
  }
}

}  // namespace

float knn_tc16_max_norm() { return 8192.f; }       // |x|^2 <= 8192: every real score stays below kPadNorm - 2 |q| |t|
int64_t knn_tc16_padded_rows(int64_t rows, bool query) { const int b = query ? kMaxUnitQ : kRows; return (rows + b - 1) / b * b; }
size_t knn_tc16_packed_bytes(int64_t rows, bool query) { return (size_t)(knn_tc16_padded_rows(rows, query) / kRows) * kTileBytes; }

cudaError_t knn_tc16_pack(const double* x, int64_t rows, int d, bool query, void* packed, float* norms, int* flags, cudaStream_t st,
                          const int* gather) {
  cudaMemsetAsync(flags, 0, 2 * sizeof(int), st);
  const int64_t rp = knn_tc16_padded_rows(rows, query);
  if (rp == 0) return cudaSuccess;
  knn_tc16_pack_kernel<<<(unsigned)((rp + 127) / 128), 128, 0, st>>>(x, rows, rp, d, query, static_cast<unsigned char*>(packed), norms,
                                                                    flags, knn_tc16_max_norm(), gather);
  return cudaGetLastError();
}

cudaError_t knn_tc16_filter(const void* qpacked, const void* tpacked, int64_t m, int64_t n, int k, const int* qflags, int* cand_idx,
                            float* cand_worst, int sm_count, cudaStream_t st, const float* thr0, const Tc16Work& work) {
  if (m == 0) return cudaSuccess;
  const int qb = work.unit_queries / kRows;
  if (work.unit_queries != qb * kRows || qb < 1 || qb > 2) return cudaErrorInvalidValue;
  const int units = (int)((m + work.unit_queries - 1) / work.unit_queries), t_tiles = (int)(knn_tc16_padded_rows(n, false) / kRows);
  auto fn = qb == 1 ? (k <= 3 ? knn_tc16_filter_kernel<5, 1> : knn_tc16_filter_kernel<kKnnCand, 1>)
                    : (k <= 3 ? knn_tc16_filter_kernel<5, 2> : knn_tc16_filter_kernel<kKnnCand, 2>);
  const size_t smem = tc_smem(qb);
  cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  const int grid = units < sm_count ? units : sm_count;
  if (work.counter) cudaMemsetAsync(work.counter, 0, sizeof(int), st);
  fn<<<grid, kTcThreads, smem, st>>>(static_cast<const unsigned char*>(qpacked), static_cast<const unsigned char*>(tpacked), m, (int)n,
                                        units, t_tiles, qflags, cand_idx, cand_worst, thr0, work);
  return cudaGetLastError();
}

}  // namespace dsp

// ---------------------------------------------------------------------------------------
// tile pruning: host plan (fit) and per-call preparation
// ---------------------------------------------------------------------------------------
namespace dsp {

namespace {

// cyclic Jacobi on a symmetric d x d matrix: a -> diagonal (eigenvalues), v = eigenvectors as columns
void jacobi_eigen(int d, double a[kPruneMaxDim][kPruneMaxDim], double v[kPruneMaxDim][kPruneMaxDim]) {
  for (int i = 0; i < d; ++i)
    for (int j = 0; j < d; ++j) v[i][j] = i == j ? 1.0 : 0.0;
  for (int sweep = 0; sweep < 100; ++sweep) {
    double off = 0.0, diag = 0.0;
    for (int p = 0; p < d; ++p) {
      diag += a[p][p] * a[p][p];
      for (int q = p + 1; q < d; ++q) off += a[p][q] * a[p][q];
    }
    if (!(off > 1e-32 * diag)) break;
    for (int p = 0; p < d; ++p)
      for (int q = p + 1; q < d; ++q) {
        if (a[p][q] == 0.0) continue;
        const double theta = (a[q][q] - a[p][p]) / (2.0 * a[p][q]);
        const double t = std::fabs(theta) > 1e150 ? 0.5 / theta : (theta >= 0 ? 1.0 : -1.0) / (std::fabs(theta) + std::sqrt(theta * theta + 1.0));
        const double c = 1.0 / std::sqrt(t * t + 1.0), s = t * c;
        for (int k = 0; k < d; ++k) { const double x = a[k][p], y = a[k][q]; a[k][p] = c * x - s * y; a[k][q] = s * x + c * y; }
        for (int k = 0; k < d; ++k) { const double x = a[p][k], y = a[q][k]; a[p][k] = c * x - s * y; a[q][k] = s * x + c * y; }
        for (int k = 0; k < d; ++k) { const double x = v[k][p], y = v[k][q]; v[k][p] = c * x - s * y; v[k][q] = s * x + c * y; }
      }
  }
}

// device scratch of one pruned call, carved in a fixed order
struct PruneScratch {
  unsigned* keys[2];
  int* vals[2];
  void* sort_tmp;
  size_t sort_bytes;
  double *ulo, *uhi, *uslack, *rad;
  int *seed, *seed_cnt, *tiles, *count[2], *ids[2], *counter;
  unsigned long long* kept;
};

// sized for the smaller unit (the most units), so one layout serves both unit sizes
size_t prune_layout(int64_t m, int64_t n, unsigned char* base, PruneScratch& s) {
  const int64_t units = (m + kRows - 1) / kRows, t_tiles = knn_tc16_padded_rows(n, false) / kRows;
  size_t b1 = 0, b2 = 0, b3 = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, b1, (const unsigned*)nullptr, (unsigned*)nullptr, (const int*)nullptr, (int*)nullptr, (int)m, 0, 30);
  cub::DeviceRadixSort::SortPairsDescending(nullptr, b2, (const int*)nullptr, (int*)nullptr, (const int*)nullptr, (int*)nullptr, (int)units);
  cub::DeviceRadixSort::SortPairsDescending(nullptr, b3, (const int*)nullptr, (int*)nullptr, (const int*)nullptr, (int*)nullptr,
                                            (int)((m + kMaxUnitQ - 1) / kMaxUnitQ));
  s.sort_bytes = std::max({b1, b2, b3});
  size_t off = 0;
  auto take = [&](size_t bytes) { void* p = base ? base + off : nullptr; off += (bytes + 255) / 256 * 256; return p; };
  for (int i = 0; i < 2; ++i) { s.keys[i] = (unsigned*)take(4 * (size_t)m); s.vals[i] = (int*)take(4 * (size_t)m); }
  s.sort_tmp = take(s.sort_bytes);
  s.ulo = (double*)take(8 * (size_t)units * kPruneMaxDim);
  s.uhi = (double*)take(8 * (size_t)units * kPruneMaxDim);
  s.uslack = (double*)take(8 * (size_t)units);
  s.rad = (double*)take(8 * (size_t)units);
  s.seed = (int*)take(4 * (size_t)units * kPruneSeedTiles);
  s.seed_cnt = (int*)take(4 * (size_t)units);
  s.tiles = (int*)take(4 * (size_t)units * t_tiles);
  for (int i = 0; i < 2; ++i) { s.count[i] = (int*)take(4 * (size_t)units); s.ids[i] = (int*)take(4 * (size_t)units); }
  s.counter = (int*)take(4);
  s.kept = (unsigned long long*)take(8);
  return off;
}

}  // namespace

void knn_prune_plan(const double* x, int64_t n, int d, KnnPrunePlan& plan) {
  KnnPruneGeom& g = plan.geom;
  std::memset(&g, 0, sizeof g);
  g.d = d;
  for (int j = 0; j < d; ++j) {
    double s = 0.0;
    for (int64_t i = 0; i < n; ++i) s += x[i * d + j];
    g.mean[j] = s / (double)n;
  }
  double cov[kPruneMaxDim][kPruneMaxDim] = {}, vec[kPruneMaxDim][kPruneMaxDim];
  for (int64_t i = 0; i < n; ++i)
    for (int p = 0; p < d; ++p)
      for (int q = p; q < d; ++q) cov[p][q] += (x[i * d + p] - g.mean[p]) * (x[i * d + q] - g.mean[q]);
  for (int p = 0; p < d; ++p)
    for (int q = p; q < d; ++q) cov[q][p] = cov[p][q] /= (double)n;
  jacobi_eigen(d, cov, vec);
  int order[kPruneMaxDim];
  std::iota(order, order + d, 0);
  std::stable_sort(order, order + d, [&](int a, int b) { return cov[a][a] > cov[b][b]; });
  for (int a = 0; a < d; ++a)
    for (int j = 0; j < d; ++j) g.axis[a][j] = vec[j][order[a]];
  // projections exactly as the device computes them (prune_project): centred features, then axis sums in feature order
  std::vector<double> pr((size_t)n * d), l1((size_t)n);
  for (int64_t i = 0; i < n; ++i) {
    double c[kPruneMaxDim], s1 = 0.0;
    for (int j = 0; j < d; ++j) { c[j] = x[i * d + j] - g.mean[j]; s1 += std::fabs(c[j]); }
    l1[(size_t)i] = s1;
    for (int a = 0; a < d; ++a) {
      double s = 0.0;
      for (int j = 0; j < d; ++j) s += c[j] * g.axis[a][j];
      pr[(size_t)i * d + a] = s;
    }
  }
  // tiles: recursive median splits along the widest axis of the range, every split on a tile boundary
  const int64_t t_tiles = knn_tc16_padded_rows(n, false) / kRows;
  plan.perm.resize((size_t)n);
  std::iota(plan.perm.begin(), plan.perm.end(), 0);
  int* perm = plan.perm.data();
  std::vector<std::pair<int64_t, int64_t>> stack{{0, t_tiles}};
  while (!stack.empty()) {
    const auto [t0, t1] = stack.back();
    stack.pop_back();
    if (t1 - t0 < 2) continue;
    const int64_t r0 = t0 * kRows, r1 = std::min<int64_t>(t1 * kRows, n), tm = t0 + (t1 - t0) / 2, rm = tm * kRows;
    int axis = 0;
    double widest = -1.0;
    for (int a = 0; a < d; ++a) {
      double lo = INFINITY, hi = -INFINITY;
      for (int64_t r = r0; r < r1; ++r) { const double v = pr[(size_t)perm[r] * d + a]; lo = std::min(lo, v); hi = std::max(hi, v); }
      if (hi - lo > widest) { widest = hi - lo; axis = a; }
    }
    std::nth_element(perm + r0, perm + rm, perm + r1, [&](int i, int j) {
      const double a = pr[(size_t)i * d + axis], b = pr[(size_t)j * d + axis];
      return a < b || (a == b && i < j);
    });
    stack.push_back({t0, tm});
    stack.push_back({tm, t1});
  }
  plan.lo.assign((size_t)t_tiles * d, INFINITY);
  plan.hi.assign((size_t)t_tiles * d, -INFINITY);
  plan.slack.assign((size_t)t_tiles, 0.0);
  for (int64_t r = 0; r < n; ++r) {
    const int64_t t = r / kRows, i = perm[r];
    for (int a = 0; a < d; ++a) {
      plan.lo[(size_t)t * d + a] = std::min(plan.lo[(size_t)t * d + a], pr[(size_t)i * d + a]);
      plan.hi[(size_t)t * d + a] = std::max(plan.hi[(size_t)t * d + a], pr[(size_t)i * d + a]);
    }
    plan.slack[(size_t)t] = std::max(plan.slack[(size_t)t], kPruneSlack * (1.0 + l1[(size_t)i]));
  }
  for (int a = 0; a < 3 && a < d; ++a) {
    double lo = INFINITY, hi = -INFINITY;
    for (int64_t t = 0; t < t_tiles; ++t) { lo = std::min(lo, plan.lo[(size_t)t * d + a]); hi = std::max(hi, plan.hi[(size_t)t * d + a]); }
    g.key_lo[a] = lo;
    g.key_scale[a] = hi > lo ? 1024.0 / (hi - lo) : 0.0;
  }
}

size_t knn_prune_scratch_bytes(int64_t m, int64_t n) {
  PruneScratch s;
  return prune_layout(m, n, nullptr, s);
}

int knn_prune_unit_queries(int64_t m, int sm_count) {
  return (m + kMaxUnitQ - 1) / kMaxUnitQ >= (int64_t)kPruneUnitsPerSm * sm_count ? kMaxUnitQ : kRows;
}

namespace {

template <int kUnitQ>
cudaError_t prune_prepare(const double* q, int64_t m, int64_t n, int d, int k, const double* train, const KnnPruneGeom* geom,
                          const int* tperm, const double* tile_lo, const double* tile_hi, const double* tile_slack, const void* tpacked,
                          void* qpacked, float* qnorm, int* qflags, const double* caller_bound, double* bound, int* cand_idx,
                          float* cand_worst, void* scratch, bool auto_fallback, int sm_count, cudaStream_t st, Tc16Work& work) {
  constexpr int kPruneThreads = kUnitQ;
  PruneScratch s;
  prune_layout(m, n, static_cast<unsigned char*>(scratch), s);
  const int units = (int)((m + kUnitQ - 1) / kUnitQ), t_tiles = (int)(knn_tc16_padded_rows(n, false) / kRows);
  const float limit = knn_tc16_max_norm();
  // query order along the curve, packed in that order
  knn_prune_keys_kernel<<<(unsigned)((m + 255) / 256), 256, 0, st>>>(q, m, geom, s.keys[0], s.vals[0]);
  size_t bytes = s.sort_bytes;
  cudaError_t e = cub::DeviceRadixSort::SortPairs(s.sort_tmp, bytes, s.keys[0], s.keys[1], s.vals[0], s.vals[1], (int)m, 0, 30, st);
  if (e != cudaSuccess) return e;
  const int* qperm = s.vals[1];
  if ((e = knn_tc16_pack(q, m, d, true, qpacked, qnorm, qflags, st, qperm)) != cudaSuccess) return e;
  knn_prune_unit_box_kernel<kPruneThreads><<<units, kPruneThreads, 0, st>>>(q, m, geom, qperm, qnorm, limit, s.ulo, s.uhi, s.uslack);
  // seed pass: each unit against its nearest tiles
  const int S = std::min(kPruneSeedTiles, t_tiles);
  knn_prune_seed_kernel<kPruneThreads><<<units, kPruneThreads, 0, st>>>(t_tiles, d, s.ulo, s.uhi, tile_lo, tile_hi, S, s.seed, s.seed_cnt);
  Tc16Work seed;
  seed.tiles = s.seed; seed.tile_count = s.seed_cnt; seed.stride = S;
  seed.qperm = qperm; seed.tperm = tperm; seed.unit_queries = kUnitQ;
  if ((e = knn_tc16_filter(qpacked, tpacked, m, n, k, qflags, cand_idx, cand_worst, sm_count, st, nullptr, seed)) != cudaSuccess) return e;
  knn_prune_bound_kernel<kPruneThreads><<<units, kPruneThreads, 0, st>>>(train, q, m, d, k, qperm, cand_idx, qnorm, limit, caller_bound, bound, s.rad);
  // tile lists, units longest first
  cudaMemsetAsync(s.kept, 0, sizeof(unsigned long long), st);
  knn_prune_list_kernel<kPruneThreads><<<units, kPruneThreads, 0, st>>>(t_tiles, d, s.ulo, s.uhi, s.uslack, s.rad, tile_lo, tile_hi, tile_slack, s.tiles,
                                                         s.count[0], s.ids[0], s.kept);
  bytes = s.sort_bytes;
  e = cub::DeviceRadixSort::SortPairsDescending(s.sort_tmp, bytes, s.count[0], s.count[1], s.ids[0], s.ids[1], units, 0, 32, st);
  if (e != cudaSuccess) return e;
  work = Tc16Work();
  work.tiles = s.tiles; work.tile_count = s.count[0]; work.stride = t_tiles;
  work.unit_order = s.ids[1]; work.counter = s.counter;
  work.kept = s.kept;
  work.kept_limit = auto_fallback ? (unsigned long long)(0.85 * (double)units * (double)t_tiles) : ~0ull;
  work.qperm = qperm; work.tperm = tperm; work.unit_queries = kUnitQ;
  return cudaGetLastError();
}

}  // namespace

cudaError_t knn_prune_prepare(const double* q, int64_t m, int64_t n, int d, int k, const double* train, const KnnPruneGeom* geom,
                              const int* tperm, const double* tile_lo, const double* tile_hi, const double* tile_slack, const void* tpacked,
                              void* qpacked, float* qnorm, int* qflags, const double* caller_bound, double* bound, int* cand_idx,
                              float* cand_worst, void* scratch, bool auto_fallback, int sm_count, cudaStream_t st, Tc16Work& work) {
  if (m == 0) return cudaSuccess;
  auto fn = knn_prune_unit_queries(m, sm_count) == kRows ? prune_prepare<kRows> : prune_prepare<kMaxUnitQ>;
  return fn(q, m, n, d, k, train, geom, tperm, tile_lo, tile_hi, tile_slack, tpacked, qpacked, qnorm, qflags, caller_bound, bound,
            cand_idx, cand_worst, scratch, auto_fallback, sm_count, st, work);
}

}  // namespace dsp
