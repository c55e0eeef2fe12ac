// match_kernels.cu — descriptor matching kernels for sm_100a and their C-ABI entry points.
//
//   scan_kernel<HammingMetric,…>   K1  brute-force Hamming k-NN          (cv::BFMatcher(NORM_HAMMING)::knnMatch,
//                                      placerec_gen_be.cpp:82-100, RelNonCentralPosSolver.cpp:303-324)
//   scan_kernel<L2Metric,…>        K2  brute-force L2 k-NN on u8 SIFT    (exact result of the FLANN call sites)
//   fused filter epilogue              placerec_gen_be.cpp:102-114
//   scan_kernel<HammingMetric,…,DM> + dm_assign_kernel
//                                  K3  DenseMatcher<LandmarkMatchingAlgorithm> (placerec_be.cpp:85-90)
//
// Layout: descriptors row-major u8 [rows][32] (ORB) / [rows][128] (SIFT quantised, exact) in HBM; the
// train side is the concatenation of candidate keyframes with a row-offset array (segments).  One CTA =
// (segment[, row split]) x (block of 128*QPT queries).  Each thread keeps QPT query descriptors and their
// k-lists in registers and scans the segment rows in ascending order from shared memory, where 8/16 KB
// tiles are staged by 1-D bulk TMA (cp.async.bulk + mbarrier, double buffered).  Every lane of a warp reads
// the same train row (shared-memory broadcast), so the kernel is bound by the INT pipe (XOR+POPC / DP4A),
// not by HBM: see DESIGN.md §"K1 roofline".
//
// Exactness: a thread scans its rows in ascending order with OpenCV's rule (strict '<' against the current
// worst, insert after equal distances), which equals "the k smallest by (distance, trainIdx)".  Row splits
// produce partial lists that are merged in split order by the same rule, so any decomposition is bit-exact.
#include <float.h>
#include <limits.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "cvb_internal.cuh"
#include "tc_match.cuh"

namespace {

constexpr int kThreads = 128;
constexpr int kStages = 2;

enum { MODE_BF = 0, MODE_DM = 1 };

struct ScanParams {
  const uint8_t* q;
  int nq;
  const uint8_t* t;
  const int32_t* seg_ptr;
  int n_seg;
  int splits;
  int chunk;  // rows per split
  int32_t* out_idx;
  void* out_dist;
  // DenseMatcher mode
  const uint8_t* skipA;
  const uint8_t* skipB;
  int ithr;
  // fused filter (k = 2, splits == 1)
  int filter;
  float thr, ratio;
  int32_t* match_train;
  float* match_dist;
  int32_t* n_matches;
};

__device__ __forceinline__ uint4 ld_nc_u4(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}

// ------------------------------------------------------------------------------------------------
// Metrics
// ------------------------------------------------------------------------------------------------
struct HammingMetric {
  static constexpr int kRowBytes = 32;
  static constexpr int kTileRows = 256;
  static constexpr bool kNeedsNorm = false;
  static constexpr bool kIsL2 = false;
  using dist_out_t = int32_t;
  struct Q {
    uint32_t w[8];
  };
  static __device__ __forceinline__ void load_q(Q& q, const uint8_t* p) {
    uint4 a = ld_nc_u4(p), b = ld_nc_u4(p + 16);
    q.w[0] = a.x; q.w[1] = a.y; q.w[2] = a.z; q.w[3] = a.w;
    q.w[4] = b.x; q.w[5] = b.y; q.w[6] = b.z; q.w[7] = b.w;
  }
  // 256-bit Hamming: FeatureMatcher::DescriptorDistanceHamming (feature_matcher_be.cpp:49-64) with the
  // SWAR bit-hack replaced by the POPC instruction.
  static __device__ __forceinline__ int dist(const Q& q, const uint4* row, int) {
    uint4 a = row[0], b = row[1];
    int d0 = __popc(q.w[0] ^ a.x) + __popc(q.w[1] ^ a.y);
    int d1 = __popc(q.w[2] ^ a.z) + __popc(q.w[3] ^ a.w);
    int d2 = __popc(q.w[4] ^ b.x) + __popc(q.w[5] ^ b.y);
    int d3 = __popc(q.w[6] ^ b.z) + __popc(q.w[7] ^ b.w);
    return (d0 + d1) + (d2 + d3);
  }
  static __device__ __forceinline__ bool less(int a, int b) { return a < b; }
  static __device__ __forceinline__ int32_t out_dist(int d) { return d; }
  static __device__ __forceinline__ float fdist(int d) { return (float)d; }
  static __device__ __forceinline__ int32_t empty_dist() { return INT_MAX; }
};

struct L2Metric {
  static constexpr int kRowBytes = 128;
  static constexpr int kTileRows = 128;
  static constexpr bool kNeedsNorm = true;
  static constexpr bool kIsL2 = true;
  using dist_out_t = float;
  struct Q {
    uint32_t w[32];
    int n2;
  };
  static __device__ __forceinline__ void load_q(Q& q, const uint8_t* p) {
    int n2 = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
      uint4 a = ld_nc_u4(p + 16 * i);
      q.w[4 * i + 0] = a.x; q.w[4 * i + 1] = a.y; q.w[4 * i + 2] = a.z; q.w[4 * i + 3] = a.w;
      n2 = __dp4a(a.x, a.x, (unsigned)n2); n2 = __dp4a(a.y, a.y, (unsigned)n2);
      n2 = __dp4a(a.z, a.z, (unsigned)n2); n2 = __dp4a(a.w, a.w, (unsigned)n2);
    }
    q.n2 = n2;
  }
  // squared L2 on u8: |a|^2 + |b|^2 - 2 a.b, all integer and exact (max 128*255^2 < 2^24)
  static __device__ __forceinline__ int dist(const Q& q, const uint4* row, int tn2) {
    unsigned acc0 = 0, acc1 = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
      uint4 a = row[i];
      acc0 = __dp4a(q.w[4 * i + 0], a.x, acc0);
      acc1 = __dp4a(q.w[4 * i + 1], a.y, acc1);
      acc0 = __dp4a(q.w[4 * i + 2], a.z, acc0);
      acc1 = __dp4a(q.w[4 * i + 3], a.w, acc1);
    }
    return q.n2 + tn2 - 2 * (int)(acc0 + acc1);
  }
  // OpenCV selects on the float distance sqrt(d2) (batch_distance.cpp): two different d2 can round to the
  // same float, which must then count as a tie.  d2a >= d2b already implies "not less".
  static __device__ __forceinline__ bool less(int a, int b) {
    return a < b && __fsqrt_rn((float)a) < __fsqrt_rn((float)b);
  }
  static __device__ __forceinline__ float out_dist(int d) { return d == INT_MAX ? FLT_MAX : __fsqrt_rn((float)d); }
  static __device__ __forceinline__ float fdist(int d) { return __fsqrt_rn((float)d); }
  static __device__ __forceinline__ float empty_dist() { return FLT_MAX; }
};

// ------------------------------------------------------------------------------------------------
// k-list updates (registers, fully unrolled)
// ------------------------------------------------------------------------------------------------
// OpenCV batchDistance rule: enter iff d < worst; placed after all entries with dist <= d.
template <class M, int K>
__device__ __forceinline__ void insert_bf(int (&wd)[K], int (&wi)[K], int d, int idx) {
  if (!M::less(d, wd[K - 1])) return;
  bool placed = false;
#pragma unroll
  for (int p = K - 1; p >= 1; --p) {
    if (!placed) {
      if (M::less(d, wd[p - 1])) {
        wd[p] = wd[p - 1];
        wi[p] = wi[p - 1];
      } else {
        wd[p] = d;
        wi[p] = idx;
        placed = true;
      }
    }
  }
  if (!placed) {
    wd[0] = d;
    wi[0] = idx;
  }
}
// DenseMatcher::listBIteration (implementation/DenseMatcher.hpp:152-176): enter iff d < worst (strict);
// std::lower_bound position, i.e. BEFORE entries with equal distance.
template <int K>
__device__ __forceinline__ void insert_dm(int (&wd)[K], int (&wi)[K], int d, int idx) {
  if (!(d < wd[K - 1])) return;
  bool placed = false;
#pragma unroll
  for (int p = K - 1; p >= 1; --p) {
    if (!placed) {
      if (!(wd[p - 1] < d)) {
        wd[p] = wd[p - 1];
        wi[p] = wi[p - 1];
      } else {
        wd[p] = d;
        wi[p] = idx;
        placed = true;
      }
    }
  }
  if (!placed) {
    wd[0] = d;
    wi[0] = idx;
  }
}

// placerec_gen_be.cpp:102-114 in float, as the reference (thresholds are float, config_backend.hpp:119-120)
__device__ __forceinline__ bool ratio_test(int i0, int i1, float dm, float dn, float thr, float ratio) {
  return i0 >= 0 && i1 >= 0 && dm <= thr && dm < __fmul_rn(ratio, dn);
}

template <class M>
constexpr size_t scan_smem_bytes() {
  return (size_t)kStages * M::kTileRows * M::kRowBytes + (size_t)kStages * M::kTileRows * sizeof(int) +
         (size_t)kStages * M::kTileRows + kStages * sizeof(uint64_t);
}

// ------------------------------------------------------------------------------------------------
// The scan kernel
// ------------------------------------------------------------------------------------------------
template <class M, int QPT, int K, int MODE>
__global__ void __launch_bounds__(kThreads) scan_kernel(const ScanParams p) {
  extern __shared__ __align__(128) uint8_t smem[];
  uint8_t* tile_base = smem;
  int* norm_base = reinterpret_cast<int*>(smem + (size_t)kStages * M::kTileRows * M::kRowBytes);
  uint8_t* skip_base = reinterpret_cast<uint8_t*>(norm_base + kStages * M::kTileRows);
  uint64_t* mbar = reinterpret_cast<uint64_t*>(skip_base + kStages * M::kTileRows);

  const int tid = threadIdx.x;
  const int seg = blockIdx.x / p.splits;
  const int split = blockIdx.x - seg * p.splits;
  const int s0 = p.seg_ptr[seg];
  const int len = p.seg_ptr[seg + 1] - s0;
  const int r0 = min(len, split * p.chunk);
  const int r1 = min(len, r0 + p.chunk);
  const int ntiles = (r1 - r0 + M::kTileRows - 1) / M::kTileRows;
  const uint8_t* tseg = p.t + (size_t)s0 * M::kRowBytes;

  // ---- queries into registers ----
  typename M::Q q[QPT];
  int wd[QPT][K], wi[QPT][K];
  bool active[QPT];
#pragma unroll
  for (int j = 0; j < QPT; j++) {
    const int qi = blockIdx.y * (kThreads * QPT) + j * kThreads + tid;
    active[j] = qi < p.nq;
    if (MODE == MODE_DM && active[j] && p.skipA) active[j] = p.skipA[qi] == 0;
    const int ql = min(qi, p.nq - 1);
    M::load_q(q[j], p.q + (size_t)ql * M::kRowBytes);
#pragma unroll
    for (int c = 0; c < K; c++) {
      wd[j][c] = (MODE == MODE_DM) ? p.ithr : INT_MAX;
      wi[j][c] = -1;
    }
  }

  // ---- TMA pipeline prologue ----
  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < kStages; s++) cvb_mbar_init(&mbar[s], 1);
    cvb_fence_mbar_init();
  }
  __syncthreads();
  auto issue = [&](int tile) {
    const int st = tile % kStages;
    const int row = r0 + tile * M::kTileRows;
    const int rows = min(M::kTileRows, r1 - row);
    const uint32_t bytes = (uint32_t)rows * M::kRowBytes;
    cvb_mbar_expect_tx(&mbar[st], bytes);
    cvb_bulk_g2s(tile_base + (size_t)st * M::kTileRows * M::kRowBytes, tseg + (size_t)row * M::kRowBytes, bytes,
                 &mbar[st]);
  };
  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < kStages; s++)
      if (s < ntiles) issue(s);
  }

  // ---- main loop over row tiles (ascending) ----
  for (int tile = 0; tile < ntiles; tile++) {
    const int st = tile % kStages;
    const uint32_t parity = (tile / kStages) & 1;
    const int row = r0 + tile * M::kTileRows;
    const int rows = min(M::kTileRows, r1 - row);
    const uint4* trow = reinterpret_cast<const uint4*>(tile_base + (size_t)st * M::kTileRows * M::kRowBytes);
    int* tnorm = norm_base + st * M::kTileRows;
    uint8_t* tskip = skip_base + st * M::kTileRows;

    if (MODE == MODE_DM && p.skipB) {  // skip flags of this tile (plain loads; u8 offsets are unaligned)
      for (int r = tid; r < rows; r += kThreads) tskip[r] = p.skipB[s0 + row + r];
    }
    cvb_mbar_wait(&mbar[st], parity);
    if (M::kNeedsNorm) {
      // |t|^2 per row; lane-rotated word order keeps the 128-B-strided reads bank-conflict free
      for (int r = tid; r < rows; r += kThreads) {
        const uint32_t* w = reinterpret_cast<const uint32_t*>(trow) + (size_t)r * (M::kRowBytes / 4);
        unsigned n2 = 0;
#pragma unroll
        for (int i = 0; i < M::kRowBytes / 4; i++) {
          uint32_t v = w[(i + tid) % (M::kRowBytes / 4)];
          n2 = __dp4a(v, v, n2);
        }
        tnorm[r] = (int)n2;
      }
    }
    if (M::kNeedsNorm || (MODE == MODE_DM && p.skipB)) __syncthreads();

    constexpr int kU4PerRow = M::kRowBytes / 16;
#pragma unroll 2
    for (int r = 0; r < rows; r++) {
      if (MODE == MODE_DM && p.skipB && tskip[r]) continue;  // warp-uniform
      const int tn2 = M::kNeedsNorm ? tnorm[r] : 0;
      const int gidx = row + r;  // segment-local trainIdx
#pragma unroll
      for (int j = 0; j < QPT; j++) {
        const int d = M::dist(q[j], trow + (size_t)r * kU4PerRow, tn2);
        if (MODE == MODE_DM) {
          if (d < wd[j][K - 1]) insert_dm<K>(wd[j], wi[j], d, gidx);
        } else {
          if (d < wd[j][K - 1]) insert_bf<M, K>(wd[j], wi[j], d, gidx);  // int pre-test, exact test inside
        }
      }
    }
    __syncthreads();  // all lanes done with this stage before it is refilled
    if (tid == 0 && tile + kStages < ntiles) issue(tile + kStages);
  }

  // ---- epilogue ----
#pragma unroll
  for (int j = 0; j < QPT; j++) {
    const int qi = blockIdx.y * (kThreads * QPT) + j * kThreads + tid;
    const bool valid = qi < p.nq;
    if (MODE == MODE_DM) {
      if (valid) {
        const size_t o = ((size_t)seg * p.nq + qi) * K;
#pragma unroll
        for (int c = 0; c < K; c++) {
          const bool has = active[j] && wi[j][c] >= 0;
          p.out_idx[o + c] = has ? wi[j][c] : -1;
          reinterpret_cast<int32_t*>(p.out_dist)[o + c] = has ? wd[j][c] : p.ithr;
        }
      }
      continue;
    }
    if (p.splits > 1) {  // partial lists, merged by merge_kernel
      if (valid) {
        const size_t o = (((size_t)seg * p.splits + split) * p.nq + qi) * K;
#pragma unroll
        for (int c = 0; c < K; c++) {
          p.out_idx[o + c] = wi[j][c];
          reinterpret_cast<int32_t*>(p.out_dist)[o + c] = wd[j][c];  // raw integer key
        }
      }
      continue;
    }
    if (p.filter) {
      bool ok = false;
      if (K >= 2 && valid) {
        const float dm = M::fdist(wd[j][0]);
        const float dn = M::fdist(wd[j][K >= 2 ? 1 : 0]);
        ok = ratio_test(wi[j][0], wi[j][K >= 2 ? 1 : 0], dm, dn, p.thr, p.ratio);
        const size_t o = (size_t)seg * p.nq + qi;
        p.match_train[o] = ok ? wi[j][0] : -1;
        p.match_dist[o] = ok ? dm : FLT_MAX;
      }
      const unsigned b = __ballot_sync(0xffffffffu, ok);
      if ((tid & 31) == 0 && b) atomicAdd(&p.n_matches[seg], __popc(b));
    } else if (valid) {
      const size_t o = ((size_t)seg * p.nq + qi) * K;
#pragma unroll
      for (int c = 0; c < K; c++) {
        p.out_idx[o + c] = wi[j][c];
        reinterpret_cast<typename M::dist_out_t*>(p.out_dist)[o + c] =
            wi[j][c] >= 0 ? M::out_dist(wd[j][c]) : M::empty_dist();
      }
    }
  }
}

// Merge the per-split partial lists of one (segment, query) in split order with the OpenCV rule.
template <class M, int K>
__global__ void merge_kernel(const int32_t* part_idx, const int32_t* part_key, int nq, int n_seg, int splits,
                             int chunk, int32_t* out_idx, void* out_dist, int filter, float thr, float ratio,
                             int32_t* match_train, float* match_dist, int32_t* n_matches) {
  const size_t gid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool valid = gid < (size_t)n_seg * nq;
  const int seg = valid ? (int)(gid / nq) : 0;
  const int qi = valid ? (int)(gid - (size_t)seg * nq) : 0;
  int wd[K], wi[K];
#pragma unroll
  for (int c = 0; c < K; c++) {
    wd[c] = INT_MAX;
    wi[c] = -1;
  }
  if (valid) {
    for (int s = 0; s < splits; s++) {
      const size_t o = (((size_t)seg * splits + s) * nq + qi) * K;
#pragma unroll
      for (int c = 0; c < K; c++) {
        const int i = part_idx[o + c];
        if (i >= 0) insert_bf<M, K>(wd, wi, part_key[o + c], i);
      }
    }
  }
  if (filter) {
    bool ok = false;
    if (valid && K >= 2) {
      const float dm = M::fdist(wd[0]), dn = M::fdist(wd[K >= 2 ? 1 : 0]);
      ok = ratio_test(wi[0], wi[K >= 2 ? 1 : 0], dm, dn, thr, ratio);
      match_train[gid] = ok ? wi[0] : -1;
      match_dist[gid] = ok ? dm : FLT_MAX;
    }
    // a warp may straddle two segments: count per lane-group by segment
    const unsigned act = __ballot_sync(0xffffffffu, ok);
    if (ok) {
      const unsigned same = __match_any_sync(act, seg);
      if ((threadIdx.x & 31) == __ffs(same) - 1) atomicAdd(&n_matches[seg], __popc(same));
    }
  } else if (valid) {
#pragma unroll
    for (int c = 0; c < K; c++) {
      out_idx[gid * K + c] = wi[c];
      reinterpret_cast<typename M::dist_out_t*>(out_dist)[gid * K + c] =
          wi[c] >= 0 ? M::out_dist(wd[c]) : M::empty_dist();
    }
  }
}

// ------------------------------------------------------------------------------------------------
// DenseMatcher::assignbest (src/dense_matcher/DenseMatcher.cpp:62-104) for A = 0,1,2,… then the final
// sweep over B (implementation/DenseMatcher.hpp:93-121).  One CTA per candidate keyframe: the k-lists and
// the pairing table live in shared memory; lane 0 runs the (inherently sequential) proposal chain, then
// the whole CTA compacts the pairings in B order.
// ------------------------------------------------------------------------------------------------
template <bool SMEM>
__global__ void __launch_bounds__(256) dm_assign_kernel(const int32_t* __restrict__ list_idx,
                                                        const int32_t* __restrict__ list_dist, int nA, int K,
                                                        const int32_t* __restrict__ seg_ptr, int ithr,
                                                        int32_t* g_vp_idx, int32_t* g_vp_dist, int32_t* outA,
                                                        int32_t* outB, float* outD, int32_t* n_out) {
  extern __shared__ __align__(16) int32_t sm[];
  __shared__ int warp_cnt[8];
  __shared__ int base_cnt;
  const int seg = blockIdx.x;
  const int s0 = seg_ptr[seg];
  const int nB = seg_ptr[seg + 1] - s0;
  const int tid = threadIdx.x;
  const int32_t* gl_i = list_idx + (size_t)seg * nA * K;
  const int32_t* gl_d = list_dist + (size_t)seg * nA * K;
  const int32_t* li;
  const int32_t* ld;
  int32_t* vp_i;
  int32_t* vp_d;
  if (SMEM) {
    int32_t* sli = sm;
    int32_t* sld = sm + (size_t)nA * K;
    vp_i = sld + (size_t)nA * K;
    vp_d = vp_i + nB;
    for (int i = tid; i < nA * K; i += blockDim.x) {
      sli[i] = gl_i[i];
      sld[i] = gl_d[i];
    }
    li = sli;
    ld = sld;
  } else {
    li = gl_i;
    ld = gl_d;
    vp_i = g_vp_idx + s0;
    vp_d = g_vp_dist + s0;
  }
  for (int b = tid; b < nB; b += blockDim.x) {
    vp_i[b] = -1;
    vp_d[b] = INT_MAX;
  }
  __syncthreads();
  if (tid == 0) {
    for (int a0 = 0; a0 < nA; a0++) {
      int a = a0, start = 0;
      for (;;) {
        bool again = false;
        for (int index = start; index < K; ++index) {
          const int b = li[a * K + index];
          if (b == -1) break;
          const int d = ld[a * K + index];
          if (vp_i[b] == -1) {
            vp_i[b] = a;
            vp_d[b] = d;
            break;
          } else if (d < vp_d[b]) {
            const int old = vp_i[b];
            vp_i[b] = a;
            vp_d[b] = d;
            a = old;
            start = 1;
            again = true;
            break;
          }
        }
        if (!again) break;
      }
    }
  }
  if (tid == 0) base_cnt = 0;
  __syncthreads();
  // ordered compaction by B index
  for (int b0 = 0; b0 < nB; b0 += blockDim.x) {
    const int b = b0 + tid;
    const bool has = b < nB && vp_i[b] != -1 && vp_d[b] < ithr;
    const unsigned bal = __ballot_sync(0xffffffffu, has);
    const int lane = tid & 31, w = tid >> 5;
    if (lane == 0) warp_cnt[w] = __popc(bal);
    __syncthreads();
    int off = base_cnt;
    for (int i = 0; i < w; i++) off += warp_cnt[i];
    if (has) {
      const int pos = s0 + off + __popc(bal & ((1u << lane) - 1));
      outA[pos] = vp_i[b];
      outB[pos] = b;
      outD[pos] = (float)vp_d[b];
    }
    __syncthreads();
    if (tid == 0) {
      int tot = 0;
      for (int i = 0; i < (int)(blockDim.x >> 5); i++) tot += warp_cnt[i];
      base_cnt += tot;
    }
    __syncthreads();
  }
  if (tid == 0) n_out[seg] = base_cnt;
}

// f32 → u8 with an integrality / range check (SIFT descriptors are integer valued 0..255)
__global__ void quantize_u8_kernel(const float* __restrict__ src, int64_t n, uint8_t* __restrict__ dst,
                                   int32_t* bad) {
  int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i >= n) return;
  bool b = false;
  if (i + 4 <= n) {
    const float4 v = *reinterpret_cast<const float4*>(src + i);
    const float f[4] = {v.x, v.y, v.z, v.w};
    uint32_t pk = 0;
#pragma unroll
    for (int c = 0; c < 4; c++) {
      const float r = rintf(f[c]);
      b |= !(r == f[c] && r >= 0.f && r <= 255.f);
      pk |= ((uint32_t)(int)fminf(fmaxf(r, 0.f), 255.f)) << (8 * c);
    }
    *reinterpret_cast<uint32_t*>(dst + i) = pk;
  } else {
    for (; i < n; i++) {
      const float r = rintf(src[i]);
      b |= !(r == src[i] && r >= 0.f && r <= 255.f);
      dst[i] = (uint8_t)(int)fminf(fmaxf(r, 0.f), 255.f);
    }
  }
  if (b) atomicOr(bad, 1);
}

// ------------------------------------------------------------------------------------------------
// Host-side planning / dispatch
// ------------------------------------------------------------------------------------------------
struct Plan {
  int qpt, splits, chunk, qblocks;
};

template <class M>
Plan make_plan(int nq, int n_seg, int max_len, int sm, int qpt_big, bool allow_split) {
  Plan pl;
  pl.qpt = qpt_big;
  pl.qblocks = (nq + kThreads * pl.qpt - 1) / (kThreads * pl.qpt);
  long ctas = (long)n_seg * pl.qblocks;
  if (ctas < 2L * sm) {
    pl.qpt = 1;
    pl.qblocks = (nq + kThreads - 1) / kThreads;
    ctas = (long)n_seg * pl.qblocks;
  }
  pl.splits = 1;
  pl.chunk = max_len > 0 ? max_len : 1;
  if (allow_split && ctas < 4L * sm && max_len > 2 * M::kTileRows) {
    long want = (4L * sm + ctas - 1) / ctas;
    long max_splits = (max_len + M::kTileRows - 1) / M::kTileRows;
    if (want > max_splits) want = max_splits;
    int chunk = (int)((max_len + want - 1) / want);
    chunk = ((chunk + M::kTileRows - 1) / M::kTileRows) * M::kTileRows;
    pl.chunk = chunk;
    pl.splits = (max_len + chunk - 1) / chunk;
  }
  return pl;
}

template <class M, int QPT, int K, int MODE>
int launch_scan(cvb_ctx* ctx, const ScanParams& sp, const Plan& pl, cudaStream_t st) {
  static cvb_once_per_device once;
  const size_t smem = scan_smem_bytes<M>();
  if (once.first(ctx->device)) {
    CVB_CUDA(ctx, cudaFuncSetAttribute(scan_kernel<M, QPT, K, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)smem));
  }
  dim3 grid((unsigned)(sp.n_seg * pl.splits), (unsigned)pl.qblocks);
  scan_kernel<M, QPT, K, MODE><<<grid, kThreads, smem, st>>>(sp);
  CVB_CHECK_LAUNCH(ctx);
  return CVB_OK;
}

template <class M, int QPT_BIG, int MODE>
int dispatch_scan(cvb_ctx* ctx, const ScanParams& sp, const Plan& pl, int k, cudaStream_t st) {
#define CVB_CASE(KK)                                                                       \
  case KK:                                                                                 \
    return pl.qpt == 1 ? launch_scan<M, 1, KK, MODE>(ctx, sp, pl, st)                      \
                       : launch_scan<M, QPT_BIG, KK, MODE>(ctx, sp, pl, st);
  switch (k) {
    CVB_CASE(1)
    CVB_CASE(2)
    CVB_CASE(3)
    CVB_CASE(4)
  }
#undef CVB_CASE
  return cvb_fail(ctx, CVB_ERR_INVALID, "k must be in 1..4 (got %d)", k);
}

template <class M, int K>
int launch_merge(cvb_ctx* ctx, const ScanParams& sp, const Plan& pl, int32_t* out_idx, void* out_dist,
                 cudaStream_t st) {
  const size_t n = (size_t)sp.n_seg * sp.nq;
  merge_kernel<M, K><<<(unsigned)((n + 255) / 256), 256, 0, st>>>(
      sp.out_idx, reinterpret_cast<const int32_t*>(sp.out_dist), sp.nq, sp.n_seg, pl.splits, pl.chunk, out_idx,
      out_dist, sp.filter, sp.thr, sp.ratio, sp.match_train, sp.match_dist, sp.n_matches);
  CVB_CHECK_LAUNCH(ctx);
  return CVB_OK;
}

int check_segs(cvb_ctx* ctx, const int32_t* h_seg_ptr, int n_seg, int* max_len, int64_t* total) {
  CVB_REQUIRE(ctx, h_seg_ptr != nullptr, "seg_ptr (host copy) is required");
  CVB_REQUIRE(ctx, n_seg >= 1, "n_seg must be >= 1");
  CVB_REQUIRE(ctx, h_seg_ptr[0] == 0, "seg_ptr[0] must be 0");
  int m = 0;
  for (int s = 0; s < n_seg; s++) {
    const int len = h_seg_ptr[s + 1] - h_seg_ptr[s];
    CVB_REQUIRE(ctx, len >= 0, "seg_ptr must be non-decreasing");
    if (len > m) m = len;
  }
  *max_len = m;
  *total = h_seg_ptr[n_seg];
  return CVB_OK;
}

// Merge of per-shard k-NN lists (map-wide k-NN with the database sharded by keyframe block over G GPUs, SURVEY §8e):
// one thread per (segment, query) row merges G lists of k by (distance, global trainIdx) — the order a single
// BFMatcher over the concatenated database produces.  Distances are compared through their int32 bit pattern, which is
// order-preserving for the non-negative floats of the L2 path and is the value itself for Hamming.
constexpr int kMaxMergeK = 8;
__global__ void shard_merge_kernel(const int32_t* __restrict__ idx_all, const int32_t* __restrict__ key_all,
                                   const int32_t* __restrict__ row_offset, int n_shards, long long n, int k,
                                   int32_t* __restrict__ out_idx, int32_t* __restrict__ out_key, int32_t empty_key) {
  const long long row = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= n) return;
  int bk[kMaxMergeK], bi[kMaxMergeK];
#pragma unroll
  for (int c = 0; c < kMaxMergeK; c++) {
    bk[c] = INT_MAX;
    bi[c] = INT_MAX;
  }
  for (int g = 0; g < n_shards; g++) {
    const int off = row_offset[g];
    const size_t o = ((size_t)g * n + row) * k;
    for (int c = 0; c < k; c++) {
      const int li = idx_all[o + c];
      if (li < 0) continue;
      int ck = key_all[o + c], ci = li + off;
#pragma unroll
      for (int s = 0; s < kMaxMergeK; s++) {   // insertion keeping (key, idx) ascending
        const bool lt = ck < bk[s] || (ck == bk[s] && ci < bi[s]);
        const int tk = bk[s], ti = bi[s];
        bk[s] = lt ? ck : tk;
        bi[s] = lt ? ci : ti;
        ck = lt ? tk : ck;
        ci = lt ? ti : ci;
      }
    }
  }
#pragma unroll
  for (int c = 0; c < kMaxMergeK; c++)
    if (c < k) {
      const bool have = bi[c] != INT_MAX;
      out_idx[row * k + c] = have ? bi[c] : -1;
      out_key[row * k + c] = have ? bk[c] : empty_key;
    }
}

// Common implementation of knn / fused-match for both metrics (device pointers).  xt / seg_tile: the resident operand
// tiles of the Hamming train rows (cvb_tc::TcParams), null when the caller has none.
template <class M, int QPT_BIG>
int knn_dev(cvb_ctx* ctx, const uint8_t* d_q, int nq, const uint8_t* d_t, const int32_t* d_seg_ptr,
            const int32_t* h_seg_ptr, int n_seg, int k, int32_t* d_idx, void* d_dist, bool filter, float thr,
            float ratio, int32_t* d_match_train, float* d_match_dist, int32_t* d_n_matches, cudaStream_t st,
            const uint8_t* xt = nullptr, const int32_t* seg_tile = nullptr) {
  CVB_REQUIRE(ctx, ctx != nullptr, "null ctx");
  CVB_REQUIRE(ctx, nq >= 0 && k >= 1 && k <= 4, "bad nq/k");
  int max_len = 0;
  int64_t total = 0;
  int rc = check_segs(ctx, h_seg_ptr, n_seg, &max_len, &total);
  if (rc) return rc;
  CVB_REQUIRE(ctx, (reinterpret_cast<uintptr_t>(d_t) & 15) == 0 && (reinterpret_cast<uintptr_t>(d_q) & 15) == 0,
              "descriptor arrays must be 16-byte aligned");
  if (filter) {
    CVB_REQUIRE(ctx, k == 2, "fused filter needs k == 2");
    CVB_CUDA(ctx, cudaMemsetAsync(d_n_matches, 0, sizeof(int32_t) * n_seg, st));
  }
  if (nq == 0) return CVB_OK;
  const cvb_tc::Formulation f = cvb_tc::choose(ctx, nq, n_seg, total, max_len, filter);
  switch (f.kind) {
    case cvb_tc::Formulation::kPerSegment: {   // tensor-core formulation (tc_match.cu), same results
      cvb_tc::TcParams tp{};
      tp.q = d_q; tp.nq = nq; tp.t = d_t; tp.seg_ptr = d_seg_ptr; tp.n_seg = n_seg;
      tp.out_idx = d_idx; tp.out_dist = d_dist; tp.filter = filter ? 1 : 0; tp.thr = thr; tp.ratio = ratio;
      tp.match_train = d_match_train; tp.match_dist = d_match_dist; tp.n_matches = d_n_matches;
      tp.h_seg = h_seg_ptr; tp.xt = xt; tp.seg_tile = seg_tile;
      return cvb_tc::launch(ctx, tp, M::kIsL2 ? 1 : 0, k, st);
    }
    case cvb_tc::Formulation::kChunked: {
      // One very long segment (map-wide k-NN): cut into uniform chunks, the tensor-core kernel on the chunks and an exact
      // merge of the chunk lists (the same (distance, index) merge that combines GPU shards).
      const int64_t chunk = f.chunk;
      const int n_ps = (int)((total + chunk - 1) / chunk);
      std::vector<int32_t> h_ps((size_t)n_ps + 1), h_off((size_t)n_ps);
      for (int c = 0; c <= n_ps; c++) h_ps[c] = (int32_t)std::min<int64_t>((int64_t)c * chunk, total);
      for (int c = 0; c < n_ps; c++) h_off[c] = (int32_t)((int64_t)c * chunk);
      // own slots: WS_TMP0/WS_TMP1 hold the quantised descriptors of the host L2 path (l2_host) at this point
      int32_t* d_ps = (int32_t*)cvb_ws(ctx, WS_CHUNK_PS, sizeof(int32_t) * (n_ps + 1));
      int32_t* d_off = (int32_t*)cvb_ws(ctx, WS_CHUNK_OFF, sizeof(int32_t) * n_ps);
      const size_t pn = (size_t)n_ps * nq * k;
      int32_t* part_i = (int32_t*)cvb_ws(ctx, WS_PART_I, pn * sizeof(int32_t));
      int32_t* part_d = (int32_t*)cvb_ws(ctx, WS_PART_D, pn * sizeof(int32_t));
      if (!d_ps || !d_off || !part_i || !part_d) return CVB_ERR_CUDA;
      CVB_CUDA(ctx, cudaMemcpyAsync(d_ps, h_ps.data(), sizeof(int32_t) * (n_ps + 1), cudaMemcpyHostToDevice, st));
      CVB_CUDA(ctx, cudaMemcpyAsync(d_off, h_off.data(), sizeof(int32_t) * n_ps, cudaMemcpyHostToDevice, st));
      CVB_CUDA(ctx, cudaStreamSynchronize(st));   // the host vectors go out of scope
      cvb_tc::TcParams tp{};
      tp.q = d_q; tp.nq = nq; tp.t = d_t; tp.seg_ptr = d_ps; tp.n_seg = n_ps;
      tp.out_idx = part_i; tp.out_dist = part_d; tp.filter = 0;
      tp.h_seg = h_ps.data();
      if ((rc = cvb_tc::launch(ctx, tp, M::kIsL2 ? 1 : 0, k, st))) return rc;
      int32_t empty_key = INT_MAX;
      if (M::kIsL2) {
        const float fmax = FLT_MAX;
        memcpy(&empty_key, &fmax, 4);
      }
      shard_merge_kernel<<<(unsigned)((nq + 255) / 256), 256, 0, st>>>(part_i, part_d, d_off, n_ps, (long long)nq, k, d_idx,
                                                                      (int32_t*)d_dist, empty_key);
      CVB_CHECK_LAUNCH(ctx);
      return CVB_OK;
    }
    case cvb_tc::Formulation::kScalar:
      break;
  }
  const Plan pl = make_plan<M>(nq, n_seg, max_len, ctx->sm_count, QPT_BIG, true);
  ScanParams sp{};
  sp.q = d_q; sp.nq = nq; sp.t = d_t; sp.seg_ptr = d_seg_ptr; sp.n_seg = n_seg;
  sp.splits = pl.splits; sp.chunk = pl.chunk;
  sp.filter = filter ? 1 : 0; sp.thr = thr; sp.ratio = ratio;
  sp.match_train = d_match_train; sp.match_dist = d_match_dist; sp.n_matches = d_n_matches;
  if (pl.splits == 1) {
    sp.out_idx = d_idx; sp.out_dist = d_dist;
    return dispatch_scan<M, QPT_BIG, MODE_BF>(ctx, sp, pl, k, st);
  }
  const size_t pn = (size_t)n_seg * pl.splits * nq * k;
  int32_t* part_i = (int32_t*)cvb_ws(ctx, WS_PART_I, pn * sizeof(int32_t));
  int32_t* part_d = (int32_t*)cvb_ws(ctx, WS_PART_D, pn * sizeof(int32_t));
  if (!part_i || !part_d) return CVB_ERR_CUDA;
  sp.out_idx = part_i; sp.out_dist = part_d;
  rc = dispatch_scan<M, QPT_BIG, MODE_BF>(ctx, sp, pl, k, st);
  if (rc) return rc;
  switch (k) {
    case 1: return launch_merge<M, 1>(ctx, sp, pl, d_idx, d_dist, st);
    case 2: return launch_merge<M, 2>(ctx, sp, pl, d_idx, d_dist, st);
    case 3: return launch_merge<M, 3>(ctx, sp, pl, d_idx, d_dist, st);
    default: return launch_merge<M, 4>(ctx, sp, pl, d_idx, d_dist, st);
  }
}

// Host wrappers validate the host seg_ptr BEFORE sizing any buffer with seg_ptr[n_seg].
int host_rows(cvb_ctx* ctx, const int32_t* seg_ptr, int n_seg, size_t* rows) {
  int max_len = 0;
  int64_t total = 0;
  int rc = check_segs(ctx, seg_ptr, n_seg, &max_len, &total);
  if (rc) return rc;
  *rows = (size_t)total;
  return CVB_OK;
}

// Host-buffer staging helper: copies q, t, seg_ptr to device workspaces.
int stage_inputs(cvb_ctx* ctx, const void* q, size_t qbytes, const void* t, size_t tbytes, const int32_t* seg_ptr,
                 int n_seg, void** d_q, void** d_t, int32_t** d_seg) {
  *d_q = cvb_ws(ctx, WS_Q, qbytes);
  *d_t = cvb_ws(ctx, WS_T, tbytes);
  *d_seg = (int32_t*)cvb_ws(ctx, WS_SEG, sizeof(int32_t) * (n_seg + 1));
  if (!*d_q || !*d_t || !*d_seg) return CVB_ERR_CUDA;
  if (qbytes) CVB_CUDA(ctx, cudaMemcpyAsync(*d_q, q, qbytes, cudaMemcpyHostToDevice, ctx->stream));
  if (tbytes) CVB_CUDA(ctx, cudaMemcpyAsync(*d_t, t, tbytes, cudaMemcpyHostToDevice, ctx->stream));
  CVB_CUDA(ctx, cudaMemcpyAsync(*d_seg, seg_ptr, sizeof(int32_t) * (n_seg + 1), cudaMemcpyHostToDevice,
                                ctx->stream));
  return CVB_OK;
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// Landmark::ComputeDescriptor (src/covins_backend/landmark_be.cpp:49-92), batched: one warp per landmark.  For every
// candidate row i the lanes hold the Hamming distances d(i, j) (j = lane, lane + 32, …; d(i,i) = 0 as in the reference's
// matrix), the median = the (int)(0.5 (n-1))-th smallest is found by a 9-step bisection over the value range [0,256]
// with ballot counts (no sort), and the first row with the strictly smallest median wins (:86-89).  HBM-bound in the
// batch (32 B per observation, read once into L1/registers); n <= 32*kLmCap candidates keep their distances in
// registers, longer lists recompute them inside the bisection.
// ------------------------------------------------------------------------------------------------
constexpr int kLmCap = 8;
__device__ __forceinline__ int ham256(const uint4& a0, const uint4& a1, const uint8_t* __restrict__ b) {
  const uint4 b0 = __ldg(reinterpret_cast<const uint4*>(b)), b1 = __ldg(reinterpret_cast<const uint4*>(b) + 1);
  return __popc(a0.x ^ b0.x) + __popc(a0.y ^ b0.y) + __popc(a0.z ^ b0.z) + __popc(a0.w ^ b0.w) + __popc(a1.x ^ b1.x) +
         __popc(a1.y ^ b1.y) + __popc(a1.z ^ b1.z) + __popc(a1.w ^ b1.w);
}
// Landmarks with at most kLmSmall observers (the common case: mean track length 8, SURVEY §8) are handled by GROUPS of 8
// lanes — four landmarks per warp, lane g of a group = candidate row g: every lane reads the group's n rows (32 B each, L1
// hits after the first lane), ranks its n distances for the median, and an 8-lane shuffle-min picks the first row with
// the strictly smallest median.  (One warp per landmark left 24 of 32 lanes idle and ran at 1.2 % of the HBM roofline.)
constexpr int kLmSmall = 8;
__global__ void __launch_bounds__(256) lm_descriptor_small_kernel(const uint8_t* __restrict__ cand, const int32_t* __restrict__ lm_ptr,
                                                                  int n_lm, int32_t* __restrict__ best_idx,
                                                                  uint8_t* __restrict__ out_desc) {
  const int l = (blockIdx.x * blockDim.x + threadIdx.x) >> 3, g = threadIdx.x & 7;
  const unsigned gmask = 0xffu << (threadIdx.x & 24);   // the 8 lanes of this group inside the warp
  if (l >= n_lm) return;
  const int o0 = lm_ptr[l], n = lm_ptr[l + 1] - o0;
  if (n > kLmSmall) return;                              // lm_descriptor_kernel (one warp per landmark) takes it
  if (n <= 0) {
    if (g == 0) best_idx[l] = -1;
    return;
  }
  const uint8_t* D = cand + (size_t)o0 * 32;
  int key = INT_MAX;
  if (g < n) {
    const uint4 a0 = __ldg(reinterpret_cast<const uint4*>(D + (size_t)g * 32)), a1 = __ldg(reinterpret_cast<const uint4*>(D + (size_t)g * 32) + 1);
    int d[kLmSmall];
#pragma unroll
    for (int j = 0; j < kLmSmall; j++) d[j] = j < n ? ham256(a0, a1, D + (size_t)j * 32) : INT_MAX;   // j == g gives 0 (matrix diagonal)
    const int kth = (int)(0.5 * (n - 1));
    int med = 0;
#pragma unroll
    for (int j = 0; j < kLmSmall; j++) {                 // the kth smallest = the value v with #{< v} <= kth < #{<= v}
      int lt = 0, le = 0;
#pragma unroll
      for (int m = 0; m < kLmSmall; m++) { lt += d[m] < d[j]; le += d[m] <= d[j]; }
      if (j < n && lt <= kth && kth < le) med = d[j];
    }
    key = (med << 3) | g;                                // smallest median, first row on ties (landmark_be.cpp:86-89)
  }
#pragma unroll
  for (int o = 4; o > 0; o >>= 1) key = min(key, __shfl_xor_sync(gmask, key, o));
  const int best = key & 7;
  if (g == 0) best_idx[l] = best;
  reinterpret_cast<uint32_t*>(out_desc + (size_t)l * 32)[g] = __ldg(reinterpret_cast<const uint32_t*>(D + (size_t)best * 32) + g);
}

__global__ void __launch_bounds__(128) lm_descriptor_kernel(const uint8_t* __restrict__ cand, const int32_t* __restrict__ lm_ptr,
                                                            int n_lm, int32_t* __restrict__ best_idx,
                                                            uint8_t* __restrict__ out_desc) {
  const int l = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (l >= n_lm) return;
  const int o0 = lm_ptr[l], n = lm_ptr[l + 1] - o0;
  if (n <= kLmSmall) return;                             // lm_descriptor_small_kernel handles it (incl. n <= 0)
  const uint8_t* D = cand + (size_t)o0 * 32;
  const int kth = (int)(0.5 * (n - 1));          // index into the sorted row, as the reference computes it
  const bool in_regs = n <= 32 * kLmCap;
  const int nc = (n + 31) >> 5;                  // 32-wide chunks of candidates actually present (warp-uniform)
  int best_med = INT_MAX, best = -1;
  for (int i = 0; i < n; i++) {
    const uint4 a0 = __ldg(reinterpret_cast<const uint4*>(D + (size_t)i * 32));
    const uint4 a1 = __ldg(reinterpret_cast<const uint4*>(D + (size_t)i * 32) + 1);
    int d[kLmCap];
    if (in_regs) {
#pragma unroll
      for (int c = 0; c < kLmCap; c++) {
        const int j = lane + 32 * c;
        d[c] = (c < nc && j < n) ? ham256(a0, a1, D + (size_t)j * 32) : INT_MAX;   // j == i gives 0, the matrix diagonal
      }
    }
    // smallest v with #{j : d(i,j) <= v} >= kth + 1
    int lo = 0, hi = 256;
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      int cnt = 0;
      if (in_regs) {
#pragma unroll
        for (int c = 0; c < kLmCap; c++)
          if (c < nc) cnt += __popc(__ballot_sync(0xffffffffu, d[c] <= mid));
      } else {
        for (int j0 = 0; j0 < n; j0 += 32) {
          const int j = j0 + lane;
          const bool le = j < n && ham256(a0, a1, D + (size_t)j * 32) <= mid;
          cnt += __popc(__ballot_sync(0xffffffffu, le));
        }
      }
      if (cnt >= kth + 1) hi = mid; else lo = mid + 1;
    }
    if (lo < best_med) { best_med = lo; best = i; }
  }
  if (lane == 0) best_idx[l] = best;
  if (lane < 8) reinterpret_cast<uint32_t*>(out_desc + (size_t)l * 32)[lane] = __ldg(reinterpret_cast<const uint32_t*>(D + (size_t)best * 32) + lane);
}

int cvb_match_hamming_tiles_dev(cvb_ctx* ctx, const uint8_t* d_q, int nq, const uint8_t* d_t, const int32_t* d_seg_ptr,
                                const int32_t* h_seg_ptr, int n_seg, float thr, float ratio, int32_t* d_match_train,
                                float* d_match_dist, int32_t* d_n_matches, const uint8_t* xt, const int32_t* seg_tile,
                                cudaStream_t st) {
  return knn_dev<HammingMetric, 4>(ctx, d_q, nq, d_t, d_seg_ptr, h_seg_ptr, n_seg, 2, nullptr, nullptr, true, thr, ratio,
                                   d_match_train, d_match_dist, d_n_matches, st, xt, seg_tile);
}

// ------------------------------------------------------------------------------------------------
// C-ABI
// ------------------------------------------------------------------------------------------------
extern "C" {

int cvb_knn_hamming_batch_dev(cvb_ctx* ctx, const uint8_t* d_q, int nq, const uint8_t* d_t,
                              const int32_t* d_seg_ptr, const int32_t* h_seg_ptr, int n_seg, int k,
                              int32_t* d_idx, int32_t* d_dist, void* stream) {
  if (!ctx) return CVB_ERR_INVALID;
  CVB_GUARD(ctx);
  return knn_dev<HammingMetric, 4>(ctx, d_q, nq, d_t, d_seg_ptr, h_seg_ptr, n_seg, k, d_idx, d_dist, false, 0.f,
                                   0.f, nullptr, nullptr, nullptr, cvb_stream(ctx, stream));
}

int cvb_match_hamming_batch_dev(cvb_ctx* ctx, const uint8_t* d_q, int nq, const uint8_t* d_t,
                                const int32_t* d_seg_ptr, const int32_t* h_seg_ptr, int n_seg, float thr,
                                float ratio, int32_t* d_match_train, float* d_match_dist, int32_t* d_n_matches,
                                void* stream) {
  if (!ctx) return CVB_ERR_INVALID;
  CVB_GUARD(ctx);
  return cvb_match_hamming_tiles_dev(ctx, d_q, nq, d_t, d_seg_ptr, h_seg_ptr, n_seg, thr, ratio, d_match_train, d_match_dist,
                                     d_n_matches, nullptr, nullptr, cvb_stream(ctx, stream));
}

int cvb_knn_hamming_batch(cvb_ctx* ctx, const uint8_t* q, int nq, const uint8_t* t, const int32_t* seg_ptr,
                          int n_seg, int k, int32_t* idx, int32_t* dist) {
  if (!ctx) return CVB_ERR_INVALID;
  CVB_GUARD(ctx);
  CVB_REQUIRE(ctx, seg_ptr && n_seg >= 1 && nq >= 0, "bad arguments");
  size_t rows = 0;
  int rc = host_rows(ctx, seg_ptr, n_seg, &rows);
  if (rc) return rc;
  void *d_q, *d_t;
  int32_t* d_seg;
  rc = stage_inputs(ctx, q, (size_t)nq * 32, t, rows * 32, seg_ptr, n_seg, &d_q, &d_t, &d_seg);
  if (rc) return rc;
  const size_t on = (size_t)n_seg * nq * k;
  int32_t* d_idx = (int32_t*)cvb_ws(ctx, WS_OUT0, on * 4);
  int32_t* d_dist = (int32_t*)cvb_ws(ctx, WS_OUT1, on * 4);
  if (!d_idx || !d_dist) return CVB_ERR_CUDA;
  rc = cvb_knn_hamming_batch_dev(ctx, (const uint8_t*)d_q, nq, (const uint8_t*)d_t, d_seg, seg_ptr, n_seg, k, d_idx,
                                 d_dist, nullptr);
  if (rc) return rc;
  if (on) {
    CVB_CUDA(ctx, cudaMemcpyAsync(idx, d_idx, on * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CVB_CUDA(ctx, cudaMemcpyAsync(dist, d_dist, on * 4, cudaMemcpyDeviceToHost, ctx->stream));
  }
  CVB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return CVB_OK;
}

int cvb_match_hamming_batch(cvb_ctx* ctx, const uint8_t* q, int nq, const uint8_t* t, const int32_t* seg_ptr,
                            int n_seg, float thr, float ratio, int32_t* match_train, float* match_dist,
                            int32_t* n_matches) {
  if (!ctx) return CVB_ERR_INVALID;
  CVB_GUARD(ctx);
  CVB_REQUIRE(ctx, seg_ptr && n_seg >= 1 && nq >= 0, "bad arguments");
  size_t rows = 0;
  int rc = host_rows(ctx, seg_ptr, n_seg, &rows);
  if (rc) return rc;
  void *d_q, *d_t;
  int32_t* d_seg;
  rc = stage_inputs(ctx, q, (size_t)nq * 32, t, rows * 32, seg_ptr, n_seg, &d_q, &d_t, &d_seg);
  if (rc) return rc;
  const size_t on = (size_t)n_seg * nq;
  int32_t* d_mt = (int32_t*)cvb_ws(ctx, WS_OUT0, on * 4);
  float* d_md = (float*)cvb_ws(ctx, WS_OUT1, on * 4);
  int32_t* d_nm = (int32_t*)cvb_ws(ctx, WS_OUT2, (size_t)n_seg * 4);
  if (!d_mt || !d_md || !d_nm) return CVB_ERR_CUDA;
  rc = cvb_match_hamming_batch_dev(ctx, (const uint8_t*)d_q, nq, (const uint8_t*)d_t, d_seg, seg_ptr, n_seg, thr,
                                   ratio, d_mt, d_md, d_nm, nullptr);
  if (rc) return rc;
  if (on) {
    CVB_CUDA(ctx, cudaMemcpyAsync(match_train, d_mt, on * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CVB_CUDA(ctx, cudaMemcpyAsync(match_dist, d_md, on * 4, cudaMemcpyDeviceToHost, ctx->stream));
  }
  CVB_CUDA(ctx, cudaMemcpyAsync(n_matches, d_nm, (size_t)n_seg * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CVB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return CVB_OK;
}

int cvb_knn_merge_shards_dev(cvb_ctx* ctx, const int32_t* d_idx_all, const void* d_dist_all, int dist_is_float,
                             const int32_t* d_row_offset, int n_shards, int64_t n, int k, int32_t* d_idx_out,
                             void* d_dist_out, void* stream) {
  if (!ctx) return CVB_ERR_INVALID;
  CVB_GUARD(ctx);
  CVB_REQUIRE(ctx, n_shards >= 1 && n >= 0 && k >= 1 && k <= kMaxMergeK, "merge_shards: need 1 <= k <= %d, n_shards >= 1",
              kMaxMergeK);
  CVB_REQUIRE(ctx, d_idx_all && d_dist_all && d_row_offset && d_idx_out && d_dist_out, "merge_shards: null buffer");
  if (n == 0) return CVB_OK;
  int32_t empty_key = INT_MAX;   // the "no neighbour" distance of the k-NN calls: INT_MAX (Hamming) / FLT_MAX (L2)
  if (dist_is_float) {
    const float fmax = FLT_MAX;
    memcpy(&empty_key, &fmax, 4);
  }
  shard_merge_kernel<<<(unsigned)((n + 255) / 256), 256, 0, cvb_stream(ctx, stream)>>>(
      d_idx_all, (const int32_t*)d_dist_all, d_row_offset, n_shards, (long long)n, k, d_idx_out, (int32_t*)d_dist_out,
      empty_key);
  CVB_CHECK_LAUNCH(ctx);
  return CVB_OK;
}

int cvb_landmark_descriptor_batch_dev(cvb_ctx* ctx, const uint8_t* d_cand, const int32_t* d_lm_ptr, int n_lm,
                                      int32_t* d_best_idx, uint8_t* d_out_desc, void* stream) {
  if (!ctx) return CVB_ERR_INVALID;
  CVB_GUARD(ctx);
  CVB_REQUIRE(ctx, n_lm >= 0 && (n_lm == 0 || (d_cand && d_lm_ptr && d_best_idx && d_out_desc)), "landmark_descriptor: bad arguments");
  CVB_REQUIRE(ctx, (reinterpret_cast<uintptr_t>(d_cand) & 15) == 0 && (reinterpret_cast<uintptr_t>(d_out_desc) & 3) == 0,
              "landmark_descriptor: misaligned buffers");
  if (n_lm == 0) return CVB_OK;
  lm_descriptor_small_kernel<<<(unsigned)(((size_t)n_lm * 8 + 255) / 256), 256, 0, cvb_stream(ctx, stream)>>>(d_cand, d_lm_ptr, n_lm,
                                                                                                            d_best_idx, d_out_desc);
  CVB_CHECK_LAUNCH(ctx);
  lm_descriptor_kernel<<<(unsigned)(((size_t)n_lm * 32 + 127) / 128), 128, 0, cvb_stream(ctx, stream)>>>(d_cand, d_lm_ptr, n_lm,
                                                                                                       d_best_idx, d_out_desc);
  CVB_CHECK_LAUNCH(ctx);
  return CVB_OK;
}

int cvb_landmark_descriptor_batch(cvb_ctx* ctx, const uint8_t* cand, const int32_t* lm_ptr, int n_lm, int32_t* best_idx,
                                  uint8_t* out_desc) {
  if (!ctx) return CVB_ERR_INVALID;
  CVB_GUARD(ctx);
  CVB_REQUIRE(ctx, n_lm >= 0 && (n_lm == 0 || (lm_ptr && best_idx && out_desc)), "landmark_descriptor: bad arguments");
  if (n_lm == 0) return CVB_OK;
  const size_t rows = (size_t)lm_ptr[n_lm];
  CVB_REQUIRE(ctx, lm_ptr[0] == 0 && (rows == 0 || cand), "landmark_descriptor: bad lm_ptr / null candidates");
  uint8_t* d_c = (uint8_t*)cvb_ws(ctx, WS_T, rows * 32);
  int32_t* d_p = (int32_t*)cvb_ws(ctx, WS_SEG, sizeof(int32_t) * ((size_t)n_lm + 1));
  int32_t* d_b = (int32_t*)cvb_ws(ctx, WS_OUT0, sizeof(int32_t) * (size_t)n_lm);
  uint8_t* d_o = (uint8_t*)cvb_ws(ctx, WS_OUT1, (size_t)n_lm * 32);
  if (!d_c || !d_p || !d_b || !d_o) return CVB_ERR_CUDA;
  if (rows) CVB_CUDA(ctx, cudaMemcpyAsync(d_c, cand, rows * 32, cudaMemcpyHostToDevice, ctx->stream));
  CVB_CUDA(ctx, cudaMemcpyAsync(d_p, lm_ptr, sizeof(int32_t) * ((size_t)n_lm + 1), cudaMemcpyHostToDevice, ctx->stream));
  // landmarks without candidates keep their descriptor (the reference returns early): pass the caller's bytes through
  CVB_CUDA(ctx, cudaMemcpyAsync(d_o, out_desc, (size_t)n_lm * 32, cudaMemcpyHostToDevice, ctx->stream));
  int rc = cvb_landmark_descriptor_batch_dev(ctx, d_c, d_p, n_lm, d_b, d_o, nullptr);
  if (rc) return rc;
  CVB_CUDA(ctx, cudaMemcpyAsync(best_idx, d_b, sizeof(int32_t) * (size_t)n_lm, cudaMemcpyDeviceToHost, ctx->stream));
  CVB_CUDA(ctx, cudaMemcpyAsync(out_desc, d_o, (size_t)n_lm * 32, cudaMemcpyDeviceToHost, ctx->stream));
  CVB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return CVB_OK;
}

int cvb_quantize_u8_dev(cvb_ctx* ctx, const float* d_src, int64_t n, uint8_t* d_dst, int32_t* d_bad, void* stream) {
  if (!ctx) return CVB_ERR_INVALID;
  CVB_GUARD(ctx);
  cudaStream_t st = cvb_stream(ctx, stream);
  CVB_REQUIRE(ctx, (reinterpret_cast<uintptr_t>(d_src) & 15) == 0 && (reinterpret_cast<uintptr_t>(d_dst) & 3) == 0,
              "quantize: misaligned buffers");
  CVB_CUDA(ctx, cudaMemsetAsync(d_bad, 0, sizeof(int32_t), st));
  if (n == 0) return CVB_OK;
  const int64_t threads = (n + 3) / 4;
  quantize_u8_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, st>>>(d_src, n, d_dst, d_bad);
  CVB_CHECK_LAUNCH(ctx);
  return CVB_OK;
}

int cvb_knn_l2_u8_batch_dev(cvb_ctx* ctx, const uint8_t* d_q, int nq, const uint8_t* d_t, const int32_t* d_seg_ptr,
                            const int32_t* h_seg_ptr, int n_seg, int dim, int k, int32_t* d_idx, float* d_dist,
                            void* stream) {
  if (!ctx) return CVB_ERR_INVALID;
  CVB_GUARD(ctx);
  if (dim != 128) return cvb_fail(ctx, CVB_ERR_UNSUPPORTED, "L2 k-NN is implemented for dim == 128 (SIFT), got %d", dim);
  return knn_dev<L2Metric, 2>(ctx, d_q, nq, d_t, d_seg_ptr, h_seg_ptr, n_seg, k, d_idx, d_dist, false, 0.f, 0.f,
                              nullptr, nullptr, nullptr, cvb_stream(ctx, stream));
}

// shared host path for cvb_knn_l2_batch / cvb_match_l2_batch
static int l2_host(cvb_ctx* ctx, const float* q, int nq, const float* t, const int32_t* seg_ptr, int n_seg, int dim,
                   int k, bool filter, float thr, float ratio, int32_t* out_i, float* out_d, int32_t* n_matches) {
  if (!ctx) return CVB_ERR_INVALID;
  CVB_GUARD(ctx);
  CVB_REQUIRE(ctx, seg_ptr && n_seg >= 1 && nq >= 0, "bad arguments");
  if (dim != 128) return cvb_fail(ctx, CVB_ERR_UNSUPPORTED, "L2 k-NN is implemented for dim == 128 (SIFT), got %d", dim);
  size_t rows = 0;
  int rc = host_rows(ctx, seg_ptr, n_seg, &rows);
  if (rc) return rc;
  void *d_qf, *d_tf;
  int32_t* d_seg;
  rc = stage_inputs(ctx, q, (size_t)nq * dim * 4, t, rows * dim * 4, seg_ptr, n_seg, &d_qf, &d_tf, &d_seg);
  if (rc) return rc;
  uint8_t* d_q8 = (uint8_t*)cvb_ws(ctx, WS_TMP0, (size_t)nq * dim);
  uint8_t* d_t8 = (uint8_t*)cvb_ws(ctx, WS_TMP1, rows * dim);
  int32_t* d_bad = (int32_t*)cvb_ws(ctx, WS_FLAG, 2 * sizeof(int32_t));
  if (!d_q8 || !d_t8 || !d_bad) return CVB_ERR_CUDA;
  rc = cvb_quantize_u8_dev(ctx, (const float*)d_qf, (int64_t)nq * dim, d_q8, d_bad, nullptr);
  if (rc) return rc;
  rc = cvb_quantize_u8_dev(ctx, (const float*)d_tf, (int64_t)rows * dim, d_t8, d_bad + 1, nullptr);
  if (rc) return rc;
  int32_t bad[2] = {0, 0};
  CVB_CUDA(ctx, cudaMemcpyAsync(bad, d_bad, sizeof(bad), cudaMemcpyDeviceToHost, ctx->stream));
  CVB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (bad[0] || bad[1])
    return cvb_fail(ctx, CVB_ERR_UNSUPPORTED,
                    "L2 descriptors must be integer-valued in [0,255] (cv::xfeatures2d::SIFT output)");
  const size_t on = (size_t)n_seg * nq * (filter ? 1 : k);
  int32_t* d_i = (int32_t*)cvb_ws(ctx, WS_OUT0, on * 4);
  float* d_d = (float*)cvb_ws(ctx, WS_OUT1, on * 4);
  int32_t* d_nm = (int32_t*)cvb_ws(ctx, WS_OUT2, (size_t)n_seg * 4);
  if (!d_i || !d_d || !d_nm) return CVB_ERR_CUDA;
  rc = knn_dev<L2Metric, 2>(ctx, d_q8, nq, d_t8, d_seg, seg_ptr, n_seg, k, d_i, d_d, filter, thr, ratio, d_i, d_d,
                            d_nm, ctx->stream);
  if (rc) return rc;
  if (on) {
    CVB_CUDA(ctx, cudaMemcpyAsync(out_i, d_i, on * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CVB_CUDA(ctx, cudaMemcpyAsync(out_d, d_d, on * 4, cudaMemcpyDeviceToHost, ctx->stream));
  }
  if (filter) CVB_CUDA(ctx, cudaMemcpyAsync(n_matches, d_nm, (size_t)n_seg * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CVB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return CVB_OK;
}

int cvb_knn_l2_batch(cvb_ctx* ctx, const float* q, int nq, const float* t, const int32_t* seg_ptr, int n_seg, int dim,
                     int k, int32_t* idx, float* dist) {
  return l2_host(ctx, q, nq, t, seg_ptr, n_seg, dim, k, false, 0.f, 0.f, idx, dist, nullptr);
}

int cvb_match_l2_batch(cvb_ctx* ctx, const float* q, int nq, const float* t, const int32_t* seg_ptr, int n_seg,
                       int dim, float thr, float ratio, int32_t* match_train, float* match_dist, int32_t* n_matches) {
  return l2_host(ctx, q, nq, t, seg_ptr, n_seg, dim, 2, true, thr, ratio, match_train, match_dist, n_matches);
}

int cvb_landmark_match_batch_dev(cvb_ctx* ctx, const uint8_t* d_A, const uint8_t* d_skipA, int nA, const uint8_t* d_B,
                                 const uint8_t* d_skipB, const int32_t* d_seg_ptr, const int32_t* h_seg_ptr,
                                 int n_seg, float thr, int num_best, int32_t* d_outA, int32_t* d_outB, float* d_outD,
                                 int32_t* d_n_out, void* stream) {
  if (!ctx) return CVB_ERR_INVALID;
  CVB_GUARD(ctx);
  cudaStream_t st = cvb_stream(ctx, stream);
  CVB_REQUIRE(ctx, num_best >= 1 && num_best <= 4, "num_best must be in 1..4");
  CVB_REQUIRE(ctx, nA >= 0, "bad nA");
  CVB_REQUIRE(ctx, thr > 0.f && thr <= 257.f, "distance threshold out of range");
  int max_len = 0;
  int64_t total = 0;
  int rc = check_segs(ctx, h_seg_ptr, n_seg, &max_len, &total);
  if (rc) return rc;
  CVB_REQUIRE(ctx, (reinterpret_cast<uintptr_t>(d_A) & 15) == 0 && (reinterpret_cast<uintptr_t>(d_B) & 15) == 0,
              "descriptor arrays must be 16-byte aligned");
  if (nA == 0) {
    CVB_CUDA(ctx, cudaMemsetAsync(d_n_out, 0, sizeof(int32_t) * n_seg, st));
    return CVB_OK;
  }
  const int ithr = (int)ceilf(thr);  // integer d: (float)d < thr  <=>  d < ceil(thr)
  const size_t ln = (size_t)n_seg * nA * num_best;
  int32_t* li = (int32_t*)cvb_ws(ctx, WS_LIST_I, ln * 4);
  int32_t* ld = (int32_t*)cvb_ws(ctx, WS_LIST_D, ln * 4);
  if (!li || !ld) return CVB_ERR_CUDA;
  Plan pl = make_plan<HammingMetric>(nA, n_seg, max_len, ctx->sm_count, 4, false);
  ScanParams sp{};
  sp.q = d_A; sp.nq = nA; sp.t = d_B; sp.seg_ptr = d_seg_ptr; sp.n_seg = n_seg;
  sp.splits = 1; sp.chunk = pl.chunk; sp.out_idx = li; sp.out_dist = ld;
  sp.skipA = d_skipA; sp.skipB = d_skipB; sp.ithr = ithr;
  rc = dispatch_scan<HammingMetric, 4, MODE_DM>(ctx, sp, pl, num_best, st);
  if (rc) return rc;
  const size_t smem = ((size_t)2 * nA * num_best + (size_t)2 * max_len) * sizeof(int32_t);
  if (smem <= 200 * 1024) {
    static size_t attr = 0;
    if (smem > attr) {
      CVB_CUDA(ctx, cudaFuncSetAttribute(dm_assign_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)(200 * 1024)));
      attr = 200 * 1024;
    }
    dm_assign_kernel<true><<<n_seg, 256, smem, st>>>(li, ld, nA, num_best, d_seg_ptr, ithr, nullptr, nullptr, d_outA,
                                                     d_outB, d_outD, d_n_out);
  } else {
    int32_t* vi = (int32_t*)cvb_ws(ctx, WS_TMP0, (size_t)total * 4);
    int32_t* vd = (int32_t*)cvb_ws(ctx, WS_TMP1, (size_t)total * 4);
    if (!vi || !vd) return CVB_ERR_CUDA;
    dm_assign_kernel<false><<<n_seg, 256, 0, st>>>(li, ld, nA, num_best, d_seg_ptr, ithr, vi, vd, d_outA, d_outB,
                                                   d_outD, d_n_out);
  }
  CVB_CHECK_LAUNCH(ctx);
  return CVB_OK;
}

int cvb_landmark_match_batch(cvb_ctx* ctx, const uint8_t* A, const uint8_t* skipA, int nA, const uint8_t* B,
                             const uint8_t* skipB, const int32_t* seg_ptr, int n_seg, float thr, int num_best,
                             int32_t* outA, int32_t* outB, float* outD, int32_t* n_out) {
  if (!ctx) return CVB_ERR_INVALID;
  CVB_GUARD(ctx);
  CVB_REQUIRE(ctx, seg_ptr && n_seg >= 1 && nA >= 0, "bad arguments");
  size_t rows = 0;
  int rc = host_rows(ctx, seg_ptr, n_seg, &rows);
  if (rc) return rc;
  void *d_A, *d_B;
  int32_t* d_seg;
  rc = stage_inputs(ctx, A, (size_t)nA * 32, B, rows * 32, seg_ptr, n_seg, &d_A, &d_B, &d_seg);
  if (rc) return rc;
  uint8_t* d_sA = nullptr;
  uint8_t* d_sB = nullptr;
  if (skipA) {
    d_sA = (uint8_t*)cvb_ws(ctx, WS_SKIPA, (size_t)nA);
    if (!d_sA) return CVB_ERR_CUDA;
    if (nA) CVB_CUDA(ctx, cudaMemcpyAsync(d_sA, skipA, (size_t)nA, cudaMemcpyHostToDevice, ctx->stream));
  }
  if (skipB) {
    d_sB = (uint8_t*)cvb_ws(ctx, WS_SKIPB, rows);
    if (!d_sB) return CVB_ERR_CUDA;
    if (rows) CVB_CUDA(ctx, cudaMemcpyAsync(d_sB, skipB, rows, cudaMemcpyHostToDevice, ctx->stream));
  }
  int32_t* d_oA = (int32_t*)cvb_ws(ctx, WS_OUT0, rows * 4);
  int32_t* d_oB = (int32_t*)cvb_ws(ctx, WS_OUT1, rows * 4);
  float* d_oD = (float*)cvb_ws(ctx, WS_OUT2, rows * 4);
  int32_t* d_n = (int32_t*)cvb_ws(ctx, WS_MISC, (size_t)n_seg * 4);
  if (!d_oA || !d_oB || !d_oD || !d_n) return CVB_ERR_CUDA;
  rc = cvb_landmark_match_batch_dev(ctx, (const uint8_t*)d_A, d_sA, nA, (const uint8_t*)d_B, d_sB, d_seg, seg_ptr,
                                    n_seg, thr, num_best, d_oA, d_oB, d_oD, d_n, nullptr);
  if (rc) return rc;
  if (rows) {
    CVB_CUDA(ctx, cudaMemcpyAsync(outA, d_oA, rows * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CVB_CUDA(ctx, cudaMemcpyAsync(outB, d_oB, rows * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CVB_CUDA(ctx, cudaMemcpyAsync(outD, d_oD, rows * 4, cudaMemcpyDeviceToHost, ctx->stream));
  }
  CVB_CUDA(ctx, cudaMemcpyAsync(n_out, d_n, (size_t)n_seg * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CVB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return CVB_OK;
}

}  // extern "C"
