// Dense KNN candidate scan on the 5th-generation tensor cores (SURVEY.md section 8 row f3).
//
// The reference's sequence-feature variant (compare_feature_methods.py:77-176) flattens per-frame
// (energy, zcr) sequences to D = 2 * max_len (hundreds to thousands) before KNeighborsClassifier --
// the one place where the query-vs-train distance is a genuinely dense contraction
// (sklearn picks brute force for D > 15, sklearn/neighbors/_base.py:615-641).
//
//   score(q, t) = |t|^2 - 2 q.t        (|q|^2 is constant per query)
//
//   pack    float64 rows -> two fp16 planes (hi = fp16(x), lo = fp16(x - hi): 22 significant bits),
//           written tile by tile in the tensor core's canonical K-major shared-memory layout
//           (8 x 16-byte core matrices, no swizzle), so one stage of the pipeline is two contiguous
//           32 KB bulk copies (cp.async.bulk, no tensor map) -- plus |x|^2 per row.
//   scan    persistent CTAs, one per block of 128 queries, three warp roles:
//             warp 0    TMA producer: 2-stage ring of {Q_hi, Q_lo} 128x64 and {T_hi, T_lo} 256x64 tiles (96 KB a stage)
//             warp 1    one thread issues tcgen05.mma (cta_group::1, kind::f16, M = 128, N = 256, K = 16):
//                       acc += Q_hi.T_hi + Q_hi.T_lo + Q_lo.T_hi into a double-buffered fp32
//                       accumulator in TMEM (2 x 256 columns); tcgen05.commit frees the ring slot
//             warps 2-5 epilogue: tcgen05.ld 32 columns at a time (one query row per thread), fused
//                       score + running top-8 candidate list in registers -- the m x n distance
//                       matrix never exists, the accumulator never leaves the SM
//   rerank  (knn.cu) float64 direct-form distances of the 8 candidates, certificate against the
//           worst kept score minus a bound on the tensor-core evaluation, float64 rescan otherwise:
//           neighbours and labels never depend on the reduced-precision scan.
#include <cuda_fp16.h>

#include "kernels.cuh"
#include "knn.cuh"
#include "ptx.cuh"

namespace dsp {

namespace {

constexpr int kBM = 128, kBN = 256, kBK = 64;          // CTA tile: queries x train rows x features per stage
constexpr int kQTileBytes = kBM * kBK * 2;               // one fp16 plane of a query tile: 16 KB
constexpr int kTTileBytes = kBN * kBK * 2;               // one fp16 plane of a train tile: 32 KB
constexpr int kStageBytes = 2 * kQTileBytes + 2 * kTTileBytes;   // Q_hi, Q_lo, T_hi, T_lo: 96 KB
constexpr int kStages = 2;
constexpr int kAccStages = 2;
constexpr int kDenseThreads = 192;
constexpr int kTmemCols = kAccStages * kBN;              // 512 fp32 columns: all of TMEM
constexpr size_t kDenseSmem = (size_t)kStages * kStageBytes + 256;
// canonical K-major, no-swizzle layout of a 128 x 64 fp16 tile: core matrix = 8 rows x 16 bytes (128 B contiguous);
// the 8 core matrices along K of one 8-row group are contiguous (LBO = 128 B), row groups follow (SBO = 1024 B)
constexpr uint32_t kLBO = 128, kSBO = 1024;
// instruction descriptor (kind::f16): D = F32 (bits 4-5 = 1), A = B = F16 (0), both K-major, N >> 3 at bit 17, M >> 4 at bit 24
constexpr uint32_t kIdesc = (1u << 4) | ((uint32_t)(kBN >> 3) << 17) | ((uint32_t)(kBM >> 4) << 24);

__device__ __forceinline__ void cand_insert8(float (&cd)[kKnnCand], int (&ci)[kKnnCand], float d, int idx) {
  if (d < cd[kKnnCand - 1]) {
    cd[kKnnCand - 1] = d; ci[kKnnCand - 1] = idx;
#pragma unroll
    for (int s = kKnnCand - 1; s > 0; --s) {
      if (cd[s] < cd[s - 1]) {
        const float td = cd[s]; cd[s] = cd[s - 1]; cd[s - 1] = td;
        const int ti = ci[s]; ci[s] = ci[s - 1]; ci[s - 1] = ti;
      }
    }
  }
}

// ---------------------------------------------------------------------------------------
// pack: one warp per (padded) row
// ---------------------------------------------------------------------------------------
__global__ void knn_dense_pack_kernel(const double* __restrict__ x, int64_t rows, int64_t rows_padded, int d, int kb_count,
                                      int block_rows, unsigned char* __restrict__ packed, float* __restrict__ norms,
                                      float pad_norm, int* __restrict__ flags) {
  const int lane = threadIdx.x & 31;
  const int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= rows_padded) return;
  const int64_t rb = r / block_rows;
  const int rr = (int)(r % block_rows), g = rr >> 3, r8 = rr & 7;
  const size_t tile_bytes = (size_t)block_rows * kBK * 2;
  double ss = 0.0;
  bool big = false;
  for (int kc_global = lane; kc_global < kb_count * 8; kc_global += 32) {
    __align__(16) __half hi[8];
    __align__(16) __half lo[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int c = kc_global * 8 + j;
      const double v = (r < rows && c < d) ? x[r * d + c] : 0.0;
      ss += v * v;
      big |= !(fabs(v) <= 60000.0);                        // fp16 range (also catches NaN): the caller falls back to float64
      const __half h = __float2half_rn((float)v);
      hi[j] = h;
      lo[j] = __float2half_rn((float)(v - (double)__half2float(h)));
    }
    const int kb = kc_global >> 3, kc = kc_global & 7;
    unsigned char* dst = packed + ((size_t)(rb * kb_count + kb) * 2) * tile_bytes + g * kSBO + kc * kLBO + r8 * 16;
    *reinterpret_cast<uint4*>(dst) = *reinterpret_cast<const uint4*>(hi);
    *reinterpret_cast<uint4*>(dst + tile_bytes) = *reinterpret_cast<const uint4*>(lo);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  big = __any_sync(0xffffffffu, big);
  if (lane == 0) {
    const float nf = r < rows ? (float)ss : pad_norm;
    norms[r] = nf;
    if (r < rows) atomicMax(&flags[0], __float_as_int(nf));      // non-negative floats order like ints
    if (big) atomicOr(&flags[1], 1);
  }
}

// ---------------------------------------------------------------------------------------
// scan
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kDenseThreads, 1)
knn_dense_scan_kernel(const unsigned char* __restrict__ qpacked, const unsigned char* __restrict__ tpacked,
                      const float* __restrict__ tnorm, int64_t m, int q_blocks, int t_blocks, int kb_count,
                      int* __restrict__ cand_idx, float* __restrict__ cand_worst) {
  extern __shared__ __align__(1024) unsigned char smem[];
  uint64_t* bar_full = reinterpret_cast<uint64_t*>(smem + (size_t)kStages * kStageBytes);
  uint64_t* bar_empty = bar_full + kStages;
  uint64_t* bar_tfull = bar_empty + kStages;
  uint64_t* bar_tempty = bar_tfull + kAccStages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar_tempty + kAccStages);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  if (tid == 0) {
    for (int i = 0; i < kStages; ++i) { mbar_init(&bar_full[i], 1); mbar_init(&bar_empty[i], 1); }
    for (int i = 0; i < kAccStages; ++i) { mbar_init(&bar_tfull[i], 1); mbar_init(&bar_tempty[i], 4); }
    mbar_fence_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t ring = smem_u32(smem);

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      int s = 0; uint32_t ph = 0;
      for (int qb = blockIdx.x; qb < q_blocks; qb += gridDim.x)
        for (int tb = 0; tb < t_blocks; ++tb)
          for (int kb = 0; kb < kb_count; ++kb) {
            mbar_wait(&bar_empty[s], ph ^ 1u);
            mbar_expect_tx(&bar_full[s], (uint32_t)kStageBytes);
            const uint32_t dst = ring + (uint32_t)s * kStageBytes;
            bulk_g2s(dst, qpacked + ((size_t)qb * kb_count + kb) * (2 * kQTileBytes), 2 * kQTileBytes, &bar_full[s]);
            bulk_g2s(dst + 2 * kQTileBytes, tpacked + ((size_t)tb * kb_count + kb) * (2 * kTTileBytes), 2 * kTTileBytes, &bar_full[s]);
            if (++s == kStages) { s = 0; ph ^= 1u; }
          }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===== MMA issuer: one thread =====
    if (lane == 0) {
      int s = 0, as = 0; uint32_t ph = 0, aph = 0;
      for (int qb = blockIdx.x; qb < q_blocks; qb += gridDim.x)
        for (int tb = 0; tb < t_blocks; ++tb) {
          mbar_wait(&bar_tempty[as], aph ^ 1u);          // the epilogue has drained this accumulator
          tc_fence_after();
          const uint32_t d_tmem = tmem_base + (uint32_t)(as * kBN);
          for (int kb = 0; kb < kb_count; ++kb) {
            mbar_wait(&bar_full[s], ph);
            tc_fence_after();
            const uint32_t q_hi = ring + (uint32_t)s * kStageBytes, q_lo = q_hi + kQTileBytes, t_hi = q_hi + 2 * kQTileBytes, t_lo = t_hi + kTTileBytes;
#pragma unroll
            for (int k4 = 0; k4 < kBK / 16; ++k4) {
              const uint32_t off = (uint32_t)k4 * 2u * kLBO;   // 16 features = two core matrices along K
              umma_f16(d_tmem, umma_desc<kLBO, kSBO>(q_hi + off), umma_desc<kLBO, kSBO>(t_hi + off), kIdesc, (uint32_t)((kb | k4) != 0));
              umma_f16(d_tmem, umma_desc<kLBO, kSBO>(q_hi + off), umma_desc<kLBO, kSBO>(t_lo + off), kIdesc, 1u);
              umma_f16(d_tmem, umma_desc<kLBO, kSBO>(q_lo + off), umma_desc<kLBO, kSBO>(t_hi + off), kIdesc, 1u);
            }
            umma_commit(&bar_empty[s]);                   // the ring slot is free once these MMAs have read it
            if (++s == kStages) { s = 0; ph ^= 1u; }
          }
          umma_commit(&bar_tfull[as]);                    // accumulator complete
          if (++as == kAccStages) { as = 0; aph ^= 1u; }
        }
    }
    __syncwarp();
  } else {
    // ===== epilogue: warps 2..5, TMEM lane group = warp % 4, one query row per thread =====
    const int lg = warp & 3;
    const int row = lg * 32 + lane;
    int as = 0; uint32_t aph = 0;
    for (int qb = blockIdx.x; qb < q_blocks; qb += gridDim.x) {
      float cd[kKnnCand]; int ci[kKnnCand];
#pragma unroll
      for (int c = 0; c < kKnnCand; ++c) { cd[c] = INFINITY; ci[c] = -1; }
      for (int tb = 0; tb < t_blocks; ++tb) {
        mbar_wait(&bar_tfull[as], aph);
        tc_fence_after();
        const uint32_t taddr = tmem_base + ((uint32_t)(lg * 32) << 16) + (uint32_t)(as * kBN);
#pragma unroll 1
        for (int c0 = 0; c0 < kBN; c0 += 32) {
          uint32_t v[32];
          tmem_ld32(taddr + (uint32_t)c0, v);
          tmem_ld_wait();
          const float4* tn4 = reinterpret_cast<const float4*>(tnorm + (size_t)tb * kBN + c0);
          const int base = tb * kBN + c0;
#pragma unroll
          for (int j4 = 0; j4 < 8; ++j4) {
            const float4 t = __ldg(tn4 + j4);
            cand_insert8(cd, ci, fmaf(-2.f, __uint_as_float(v[4 * j4 + 0]), t.x), base + 4 * j4 + 0);
            cand_insert8(cd, ci, fmaf(-2.f, __uint_as_float(v[4 * j4 + 1]), t.y), base + 4 * j4 + 1);
            cand_insert8(cd, ci, fmaf(-2.f, __uint_as_float(v[4 * j4 + 2]), t.z), base + 4 * j4 + 2);
            cand_insert8(cd, ci, fmaf(-2.f, __uint_as_float(v[4 * j4 + 3]), t.w), base + 4 * j4 + 3);
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bar_tempty[as]);
        if (++as == kAccStages) { as = 0; aph ^= 1u; }
      }
      const int64_t q = (int64_t)qb * kBM + row;
      if (q < m) {
#pragma unroll
        for (int c = 0; c < kKnnCand; ++c) cand_idx[q * kKnnCand + c] = ci[c];
        cand_worst[q] = cd[kKnnCand - 1];
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

}  // namespace

int knn_dense_kblocks(int d) { return (d + kBK - 1) / kBK; }
int knn_dense_block_rows(bool train) { return train ? kBN : kBM; }
int64_t knn_dense_padded_rows(int64_t rows, bool train) {
  const int b = knn_dense_block_rows(train);
  return (rows + b - 1) / b * b;
}
size_t knn_dense_packed_bytes(int64_t rows, int d, bool train) {
  return (size_t)knn_dense_padded_rows(rows, train) * (size_t)knn_dense_kblocks(d) * kBK * 2 * 2;
}

cudaError_t knn_dense_pack(const double* x, int64_t rows, int d, bool train, void* packed, float* norms, float pad_norm,
                           int* flags, bool reset_flags, cudaStream_t st) {
  const int64_t rows_padded = knn_dense_padded_rows(rows, train);
  if (reset_flags) cudaMemsetAsync(flags, 0, 2 * sizeof(int), st);
  if (rows_padded == 0) return cudaSuccess;
  const int warps = 8;
  knn_dense_pack_kernel<<<(unsigned)((rows_padded + warps - 1) / warps), warps * 32, 0, st>>>(
      x, rows, rows_padded, d, knn_dense_kblocks(d), knn_dense_block_rows(train), static_cast<unsigned char*>(packed), norms,
      pad_norm, flags);
  return cudaGetLastError();
}

cudaError_t knn_dense_scan(const void* qpacked, const void* tpacked, const float* tnorm, int64_t m, int64_t n, int d,
                           int* cand_idx, float* cand_worst, int sm_count, cudaStream_t st) {
  if (m == 0) return cudaSuccess;
  const int q_blocks = (int)(knn_dense_padded_rows(m, false) / kBM), t_blocks = (int)(knn_dense_padded_rows(n, true) / kBN);
  cudaError_t e = cudaFuncSetAttribute(knn_dense_scan_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kDenseSmem);
  if (e != cudaSuccess) return e;
  const int grid = q_blocks < sm_count ? q_blocks : sm_count;
  knn_dense_scan_kernel<<<grid, kDenseThreads, kDenseSmem, st>>>(static_cast<const unsigned char*>(qpacked),
                                                                 static_cast<const unsigned char*>(tpacked), tnorm, m, q_blocks,
                                                                 t_blocks, knn_dense_kblocks(d), cand_idx, cand_worst);
  return cudaGetLastError();
}

}  // namespace dsp
