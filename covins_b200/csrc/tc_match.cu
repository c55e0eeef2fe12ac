// tc_match.cu — descriptor k-NN on the 5th-generation tensor cores (tcgen05, kind::i8, accumulators in TMEM).
//
// Same contract as scan_kernel in match_kernels.cu (K1 Hamming / K2 L2 with the OpenCV k-NN rule, optional fused ratio
// filter), different bound.  The POPC formulation tops out at 16 POPC/clk/SM (measured: 94 % of that roofline).  Here the
// pairwise term is an 8-bit GEMM issued as tcgen05.mma.cta_group::1.kind::i8 (M = 128 queries, N = 128 train rows, K = 32
// bytes per instruction), the query block held in tensor memory for the CTA's lifetime and 128x128 s32 accumulators in
// tensor memory.  One TMEM lane = one query row = one epilogue thread, which receives the train rows of a segment in
// ascending order — so the per-query selection is the same sequential OpenCV rule as in the scalar kernel and the result is
// bit-identical.  A CTA owns one block of 128 queries and streams a contiguous range of candidate segments.  Two kernels:
//
// tc_scan_kernel<K>: L2 on u8 SIFT rows, |a-b|^2 = |a|^2 + |b|^2 - 2 <a, b> (exact in s32).  Warp-specialised, persistent
// (one CTA per SM):
//   warps 0-15   epilogue   4 column groups x 4 warps: wait tfull[s] → tcgen05.ld 32x32b.x32 → d = |q|^2 + |t|^2 - 2 acc →
//                           sqrtf key → k-list → tempty[s]; at a segment's end the 4 group lists of a query are merged
//   warps 16-23  producers  two threads per train row: 16-B loads of the packed rows (two tiles in flight in registers) →
//                           canonical K-major no-swizzle UMMA layout in a 4-stage ring + row norms → fence.proxy.async → full[s]
//   warp 24      MMA        wait full[s] and a free accumulator → 4 x tcgen05.mma into a 3-stage TMEM ring → tcgen05.commit
//
// xt::tc_xt_kernel<K>: Hamming on 256-bit ORB rows from operand tiles expanded once, with the distance folded into the GEMM
// (namespace xt below).
#include <float.h>
#include <limits.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "cvb_internal.cuh"
#include "tc_match.cuh"

namespace cvb_tc {

constexpr int TM = 128;       // queries per CTA (UMMA M)
constexpr int TN = 128;       // train rows per tile (UMMA N)
constexpr int STAGES = 4;        // shared-memory ring of train tiles
constexpr int ACC_STAGES = 3;    // TMEM ring of 128-column accumulators: columns [0, 384); the query operand sits at column 384
constexpr uint32_t A_COL = ACC_STAGES * 128;
constexpr int NORM_RING = 8;
constexpr int kInf = 0x3FFFFFFF;   // list sentinel; rows that must never enter carry this as their norm term

// ---- mbarrier / tcgen05 wrappers -------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(cvb_smem_addr(bar)) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n"
      ".reg .pred P;\n"
      "elect.sync _|P, 0xffffffff;\n"
      "selp.b32 %0, 1, 0, P;\n"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(cvb_smem_addr(bar))
               : "memory");
}
__device__ __forceinline__ void tc_mma_i8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
      : "memory");
}
// A operand from tensor memory (row i of the 128 x K block in lane i, four K bytes per 32-bit column): the query block
// is constant for the CTA's lifetime, and with both operands in shared memory the operand fetch alone (8 KB per 64-cycle
// instruction) saturates the 128 B/clk shared-memory port that the producers' stores also need.
__device__ __forceinline__ void tc_mma_i8_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], [%1], %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(acc)
      : "memory");
}
// 32 lanes x 8 columns per call: thread t of the warp writes registers r[0..7] to lane (warp % 4) * 32 + t
__device__ __forceinline__ void tc_st8(uint32_t taddr, const uint32_t* r) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]),
               "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
__device__ __forceinline__ void tc_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
        "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// 32 lanes x 128 columns, the low 16 bits of two adjacent columns packed into one register (even column low, odd column high)
__device__ __forceinline__ void tc_ld64_pack16(uint32_t taddr, uint32_t (&r)[64]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.pack::16b.x64.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,"
      "%32,%33,%34,%35,%36,%37,%38,%39,%40,%41,%42,%43,%44,%45,%46,%47,%48,%49,%50,%51,%52,%53,%54,%55,%56,%57,%58,%59,%60,%61,%62,%63}, [%64];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
        "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31]), "=r"(r[32]), "=r"(r[33]), "=r"(r[34]), "=r"(r[35]), "=r"(r[36]),
        "=r"(r[37]), "=r"(r[38]), "=r"(r[39]), "=r"(r[40]), "=r"(r[41]), "=r"(r[42]), "=r"(r[43]), "=r"(r[44]), "=r"(r[45]),
        "=r"(r[46]), "=r"(r[47]), "=r"(r[48]), "=r"(r[49]), "=r"(r[50]), "=r"(r[51]), "=r"(r[52]), "=r"(r[53]), "=r"(r[54]),
        "=r"(r[55]), "=r"(r[56]), "=r"(r[57]), "=r"(r[58]), "=r"(r[59]), "=r"(r[60]), "=r"(r[61]), "=r"(r[62]), "=r"(r[63])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// shared-memory matrix descriptor: K-major, no swizzle (canonical layout ((8,n),2):((16 B, SBO), LBO)); version 1
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;   // descriptor version (Blackwell)
  return d;                 // base_offset 0, lbo_mode 0, layout_type 0 (SWIZZLE_NONE)
}
// instruction descriptor, kind::i8: D = s32 (2), A = B = u8 (0), both K-major, N >> 3 at [17,23), M >> 4 at [24,29)
__device__ __forceinline__ uint32_t make_idesc() {
  return (2u << 4) | (0u << 7) | (0u << 10) | ((uint32_t)(TN >> 3) << 17) | ((uint32_t)(TM >> 4) << 24);
}

__device__ __forceinline__ uint4 ldg_nc(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}

// k-list of (key, idx) kept sorted ascending by (key, idx); OpenCV rule for a stream with ascending idx:
// enter iff key < worst key; placed after all entries with key <= new key.
template <int K>
__device__ __forceinline__ void insert_key(int (&wk)[K], int (&wi)[K], int key, int idx) {
  if (!(key < wk[K - 1])) return;
  bool placed = false;
#pragma unroll
  for (int p = K - 1; p >= 1; --p) {
    if (!placed) {
      if (key < wk[p - 1]) { wk[p] = wk[p - 1]; wi[p] = wi[p - 1]; }
      else { wk[p] = key; wi[p] = idx; placed = true; }
    }
  }
  if (!placed) { wk[0] = key; wi[0] = idx; }
}
// merge rule for partial lists of disjoint row subsets: k smallest by (key, idx)
template <int K>
__device__ __forceinline__ void insert_lex(int (&wk)[K], int (&wi)[K], int key, int idx) {
  auto lt = [](int k1, int i1, int k2, int i2) { return k1 < k2 || (k1 == k2 && (unsigned)i1 < (unsigned)i2); };
  if (!lt(key, idx, wk[K - 1], wi[K - 1])) return;
  bool placed = false;
#pragma unroll
  for (int p = K - 1; p >= 1; --p) {
    if (!placed) {
      if (lt(key, idx, wk[p - 1], wi[p - 1])) { wk[p] = wk[p - 1]; wi[p] = wi[p - 1]; }
      else { wk[p] = key; wi[p] = idx; placed = true; }
    }
  }
  if (!placed) { wk[0] = key; wi[0] = idx; }
}

constexpr int GROUPS = 4;                       // epilogue column groups: group g owns columns [32 g, 32 g + 32) of every tile
constexpr int EPI_THREADS = 128 * GROUPS;       // 16 epilogue warps
constexpr int PROD_WARP0 = EPI_THREADS / 32;    // producer warps 16..23 (two threads per train row)
constexpr int PROD_THREADS = 256;
constexpr int MMA_WARP = PROD_WARP0 + PROD_THREADS / 32;   // warp 24
constexpr int NUM_THREADS = (MMA_WARP + 1) * 32;
constexpr int KB = 128;                         // bytes per SIFT row = operand bytes per row (u8, used as they are)
constexpr int PF = 2;                           // tiles in flight per producer thread

template <int K>
constexpr size_t smem_bytes() {
  return (size_t)STAGES * TN * KB + (size_t)NORM_RING * TN * sizeof(int) +
         (size_t)2 * TM * GROUPS * K * 2 * sizeof(int) + 64 * sizeof(uint64_t);
}

// operand row r of a tile: byte offset of its chunk 0
__device__ __forceinline__ uint32_t row_offset(int r) {
  return (uint32_t)(r >> 3) * (KB * 8) + (uint32_t)(r & 7) * 16;
}

// keys: the bit pattern of sqrtf(d2) (non-negative floats order like their bits), which is what OpenCV compares.  kInfKey
// is larger than any real key.
constexpr int kInfKey = 0x7F000000;

template <int K>
__global__ void __launch_bounds__(NUM_THREADS, 1) tc_scan_kernel(const TcParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* sB = smem;
  int* sNorm = reinterpret_cast<int*>(sB + (size_t)STAGES * TN * KB);
  int* sList = sNorm + NORM_RING * TN;                       // [2][TM][GROUPS][K][2]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sList + 2 * TM * GROUPS * K * 2);
  uint64_t* full = bars;                 // [STAGES] producers → MMA (one arrival per producer warp)
  uint64_t* empty = bars + STAGES;       // [STAGES] MMA completion → producers (tcgen05.commit)
  uint64_t* tfull = bars + 2 * STAGES;   // [ACC_STAGES] MMA completion → epilogue (tcgen05.commit)
  uint64_t* tempty = bars + 3 * STAGES;  // [ACC_STAGES] epilogue → MMA (one arrival per epilogue warp)
  __shared__ uint32_t tmem_base_s;
  __shared__ int sQNorm[TM];

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int qb = blockIdx.x % p.nqb, part = blockIdx.x / p.nqb;
  const int seg0 = (int)((long)part * p.n_seg / p.parts), seg1 = (int)((long)(part + 1) * p.n_seg / p.parts);

  // ---- one-time setup: barriers, TMEM, the query operand ----
  if (tid == 0) {
    for (int s = 0; s < STAGES; s++) {
      cvb_mbar_init(&full[s], PROD_THREADS / 32);     // one arrival per producer warp
      cvb_mbar_init(&empty[s], 1);
      cvb_mbar_init(&tfull[s], 1);
      cvb_mbar_init(&tempty[s], EPI_THREADS / 32);    // one arrival per epilogue warp
    }
    cvb_fence_mbar_init();
  }
  if (warp == MMA_WARP) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(cvb_smem_addr(&tmem_base_s)));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;
  if (tid < TM) {
    // the query block → tensor memory: thread = row = TMEM lane (warps 0-3 own lanes 32 w .. 32 w + 31), 8 columns
    // (= one K = 32 instruction's worth) per tcgen05.st
    const int q = qb * TM + tid;
    uint32_t w[32];
    unsigned nrm = 0;
    if (q < p.nq) {
#pragma unroll
      for (int c = 0; c < 8; c++) {
        const uint4 v = ldg_nc(p.q + (size_t)q * KB + 16 * c);
        w[4 * c] = v.x; w[4 * c + 1] = v.y; w[4 * c + 2] = v.z; w[4 * c + 3] = v.w;
        nrm = __dp4a(v.x, v.x, nrm); nrm = __dp4a(v.y, v.y, nrm); nrm = __dp4a(v.z, v.z, nrm); nrm = __dp4a(v.w, v.w, nrm);
      }
    } else {
#pragma unroll
      for (int i = 0; i < 32; i++) w[i] = 0;
    }
    sQNorm[tid] = (int)nrm;
    const uint32_t a_taddr = tmem_base + ((uint32_t)(warp * 32) << 16) + A_COL;
#pragma unroll
    for (int i = 0; i < KB / 32; i++) tc_st8(a_taddr + 8 * i, w + 8 * i);
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();

  if (warp >= PROD_WARP0 && warp < MMA_WARP) {
    // =================================== producers ===================================
    // Two threads per train row, 64 bytes each; the packed rows of the next PF tiles are held in registers so that the
    // HBM latency (~1 us) of a tile overlaps the stores of the previous ones.
    const int pt = tid - PROD_WARP0 * 32;   // 0..255
    const int prow = (pt & 7) | ((pt >> 4) << 3), half = (pt >> 3) & 1;
    struct TileIt {
      int seg, r0, s_begin, len, seg1;
      const int32_t* sp;
      bool done;
      __device__ void next_seg() {
        do {
          seg++;
          if (seg >= seg1) { done = true; return; }
          s_begin = sp[seg];
          len = sp[seg + 1] - s_begin;
        } while (len == 0);
        r0 = 0;
      }
      __device__ void advance() { r0 += TN; if (r0 >= len) next_seg(); }
    };
    TileIt it{seg0 - 1, 0, 0, 0, seg1, p.seg_ptr, false}, ld = it;
    it.next_seg();
    ld.next_seg();
    uint4 pf[PF][4];
    auto issue_load = [&](uint4 (&v)[4]) {
      if (!ld.done) {
        const int row = ld.r0 + prow;
        if (row < ld.len) {
          const uint8_t* src = p.t + (size_t)(ld.s_begin + row) * KB + 64 * half;
#pragma unroll
          for (int c = 0; c < 4; c++) v[c] = ldg_nc(src + 16 * c);
        }
        ld.advance();
      }
    };
#pragma unroll
    for (int u = 0; u < PF; u++) issue_load(pf[u]);
    int n = 0;
    while (!it.done) {
#pragma unroll
      for (int u = 0; u < PF; u++) {
        if (it.done) break;
        uint4 cur[4];
#pragma unroll
        for (int c = 0; c < 4; c++) cur[c] = pf[u][c];
        issue_load(pf[u]);   // refill this register slot with the tile PF steps ahead
        const int s = n % STAGES;
        if (n >= STAGES) cvb_mbar_wait(&empty[s], ((n / STAGES) - 1) & 1);
        uint8_t* dst = sB + (size_t)s * TN * KB + row_offset(prow);
        const bool rv = it.r0 + prow < it.len;
        int part = 0;   // |row|^2 over this thread's half
        if (rv) {
          unsigned n2 = 0;
#pragma unroll
          for (int c = 0; c < 4; c++) {
            n2 = __dp4a(cur[c].x, cur[c].x, n2); n2 = __dp4a(cur[c].y, cur[c].y, n2); n2 = __dp4a(cur[c].z, cur[c].z, n2); n2 = __dp4a(cur[c].w, cur[c].w, n2);
            *reinterpret_cast<uint4*>(dst + (4 * half + c) * 128) = cur[c];
          }
          part = (int)n2;
        } else {
          for (int c = 0; c < 4; c++) *reinterpret_cast<uint4*>(dst + (4 * half + c) * 128) = make_uint4(0, 0, 0, 0);
        }
        part += __shfl_xor_sync(0xffffffffu, part, 8);   // the two halves of a row sit 8 lanes apart
        if (half == 0) sNorm[(n % NORM_RING) * TN + prow] = rv ? part : kInf;   // tail rows never enter a list
        // every lane makes its own stores visible to the async proxy; ONE arrival per warp (hundreds of same-address
        // mbarrier arrivals per tile serialise in shared memory and cost more than the tile's MMAs)
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(&full[s]);
        it.advance();
        n++;
      }
    }
  } else if (warp == MMA_WARP) {
    // =================================== MMA issuer ===================================
    // The WHOLE warp walks the tile sequence with warp-uniform values and one elected lane issues: under a divergent
    // `if (lane == 0)` the compiler cannot keep the descriptors in uniform registers and wraps every tcgen05.mma in an
    // ELECT / R2UR.BROADCAST waterfall loop (~150 cycles per instruction against the 64-cycle tensor floor).
    const uint32_t idesc = make_idesc();
    const uint32_t a_tmem = tmem_base + A_COL;
    const uint32_t b_addr0 = cvb_smem_addr(sB);
    int n = 0;
    for (int seg = seg0; seg < seg1; seg++) {
      const int len = __shfl_sync(0xffffffffu, p.seg_ptr[seg + 1] - p.seg_ptr[seg], 0);
#pragma unroll 2   // left alone, the compiler unrolls this small body 4x and emits 7 copies of the issue sequence
      for (int r0 = 0; r0 < len; r0 += TN, n++) {
        const int s = n % STAGES, ts = n % ACC_STAGES;
        cvb_mbar_wait(&full[s], (n / STAGES) & 1);
        if (n >= ACC_STAGES) cvb_mbar_wait(&tempty[ts], ((n / ACC_STAGES) - 1) & 1);
        tc_fence_after();
        const uint64_t b_desc0 = make_desc(b_addr0 + (uint32_t)s * (TN * KB), 128, KB * 8);
        const uint32_t d_tmem = tmem_base + (uint32_t)ts * TN;
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < KB / 32; k++)   // K chunk k: 256 B further in shared memory (+16 in the address field), 8 columns in TMEM
            tc_mma_i8_ts(d_tmem, a_tmem + 8 * k, b_desc0 + (uint64_t)(k * 16), idesc, k > 0 ? 1u : 0u);
          tc_commit(&empty[s]);    // shared-memory slot reusable once these MMAs have read it
          tc_commit(&tfull[ts]);   // accumulator ready
        }
        __syncwarp();
      }
    }
  } else {
    // =================================== epilogue (warps 0..15) ===================================
    const int grp = warp >> 2;                  // column group
    const int row = (warp & 3) * 32 + lane;     // TMEM lane = query row inside the block
    const int q = qb * TM + row;
    const bool valid = q < p.nq;
    const int qn = sQNorm[row];
    int wk[K], wi[K], wd2[K];                   // key, index, raw integer distance (pre-test only)
    int n = 0, segc = 0;
    for (int seg = seg0; seg < seg1; seg++, segc++) {
      const int len = p.seg_ptr[seg + 1] - p.seg_ptr[seg];
#pragma unroll
      for (int c = 0; c < K; c++) { wk[c] = kInfKey; wi[c] = -1; wd2[c] = kInf; }
      for (int r0 = 0; r0 < len; r0 += TN, n++) {
        const int s = n % ACC_STAGES;
        cvb_mbar_wait(&tfull[s], (n / ACC_STAGES) & 1);
        tc_fence_after();
        const uint32_t taddr = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)s * TN + grp * 32;
        uint32_t acc[32];
        tc_ld32(taddr, acc);
        if (valid) {
          const int4* nrm4 = reinterpret_cast<const int4*>(sNorm + (n % NORM_RING) * TN + grp * 32);
#pragma unroll
          for (int i4 = 0; i4 < 8; i4++) {
            const int4 nn = nrm4[i4];
            const int nv[4] = {nn.x, nn.y, nn.z, nn.w};
#pragma unroll
            for (int j = 0; j < 4; j++) {
              const int i = 4 * i4 + j;
              const int d = qn + nv[j] - 2 * (int)acc[i];
              if (d < wd2[K - 1]) {
                const int key = __float_as_int(__fsqrt_rn((float)d));
                if (key < wk[K - 1]) {
                  insert_key<K>(wk, wi, key, r0 + grp * 32 + i);
                  const float f = __int_as_float(wk[K - 1]);   // raw-distance bound of the worst entry (pre-test)
                  wd2[K - 1] = wk[K - 1] == kInfKey ? kInf : (int)ceilf(f * f * 1.000001f) + 1;
                }
              }
            }
          }
        }
        // accumulator and norms consumed: the MMA warp may overwrite this TMEM stage
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tempty[s]);
      }
      // ---- segment finished: combine the 4 column-group lists of each query (k smallest by (key, idx)) ----
      int* lst = sList + (size_t)(segc & 1) * TM * GROUPS * K * 2;
#pragma unroll
      for (int c = 0; c < K; c++) {
        lst[((row * GROUPS + grp) * K + c) * 2 + 0] = wk[c];
        lst[((row * GROUPS + grp) * K + c) * 2 + 1] = wi[c];
      }
      asm volatile("bar.sync 1, %0;" ::"n"(EPI_THREADS) : "memory");
      if (grp == 0) {
#pragma unroll
        for (int c = 0; c < K; c++) { wk[c] = kInfKey; wi[c] = -1; }
        for (int g2 = 0; g2 < GROUPS; g2++)
#pragma unroll
          for (int c = 0; c < K; c++) {
            const int kk = lst[((row * GROUPS + g2) * K + c) * 2], ii = lst[((row * GROUPS + g2) * K + c) * 2 + 1];
            if (ii >= 0) insert_lex<K>(wk, wi, kk, ii);
          }
        float fd[K];   // final distances as float (DMatch::distance)
#pragma unroll
        for (int c = 0; c < K; c++) fd[c] = __int_as_float(wk[c]);
        if (p.filter) {
          bool ok = false;
          if (K >= 2 && valid) {
            const float dm = fd[0], dn = fd[K >= 2 ? 1 : 0];
            ok = wi[0] >= 0 && wi[K >= 2 ? 1 : 0] >= 0 && dm <= p.thr && dm < __fmul_rn(p.ratio, dn);
            const size_t o = (size_t)seg * p.nq + q;
            p.match_train[o] = ok ? wi[0] : -1;
            p.match_dist[o] = ok ? dm : FLT_MAX;
          }
          const unsigned b = __ballot_sync(0xffffffffu, ok);
          if (lane == 0 && b) atomicAdd(&p.n_matches[seg], __popc(b));
        } else if (valid) {
          const size_t o = ((size_t)seg * p.nq + q) * K;
#pragma unroll
          for (int c = 0; c < K; c++) {
            p.out_idx[o + c] = wi[c];
            reinterpret_cast<float*>(p.out_dist)[o + c] = wi[c] >= 0 ? fd[c] : FLT_MAX;
          }
        }
      }
    }
  }
  // ---- teardown ----
  tc_fence_before();
  __syncthreads();
  if (warp == MMA_WARP) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base));
  }
}

// ===================================================================================================================
// Hamming k-NN on PRE-EXPANDED operand tiles.
//
// Hamming(a,b) = popc(a) + popc(b) - 2 popc(a & b), and popc(a & b) is an 8-bit GEMM once the 256 bits of a row are
// expanded to bytes.  Expanding inside the matching kernel costs >= 64 logic operations per row and tile, and rebuilding
// the distance from the accumulator costs ALU work per pair in the epilogue: the ALU, not the tensor pipe, then bounds
// the kernel.  Both disappear when the operand the tensor core reads is stored once and reused by every query:
//
//   * cvb_tc::expand_tiles writes, per keyframe, ceil(rows / 128) tiles of 128 rows x 288 operand bytes in exactly the
//     shared-memory image tcgen05.mma wants (K-major, no swizzle, 8-row groups of 2304 B): 256 data bytes (0x80 = -128
//     as s8 for a set bit) + a 32-byte KEY slice.  A tile is 36 KB and contiguous, so the producer is ONE thread issuing
//     cp.async.bulk copies (TMA engine) — no register path, no expansion in the matching kernel.  The map database
//     (map_db.cu) keeps these tiles resident next to the packed rows; 9 bytes of HBM per descriptor byte, read at
//     ~2 TB/s by a kernel that is bound by the tensor pipe, not by HBM.  A train set without resident tiles (the
//     raw-pointer API) is expanded into the workspace by launch() before the matching kernel runs.
//   * the key slice folds the whole distance into the GEMM: with query bytes 0/2 (u8) and
//         A key bytes = [1, 128, 128, 128, c4, c5, c6, 0...]   c4 + c5 + c6 = 2 popc(q)      (per query row)
//         B key bytes = [col, p1, p2, p3, 64, 64, 64, 0...]    p1 + p2 + p3 = popc(t)        (per train row)
//     the s32 accumulator is  (popc(q) + popc(t) - 2 popc(q & t)) << 7 | col  =  Hamming << 7 | row-in-tile: the sort key
//     itself, <= 32895, so the epilogue reads it as packed 16-bit pairs (LDTM.PACK16BIT) and runs nothing but the
//     packed min/max network.  Rows past a keyframe's end carry B key bytes [127,127,127,127,0...] → key 48895, which
//     never enters a list.
//   * three segment STREAMS: epilogue group g (4 warps = the 128 TMEM lanes) owns accumulator g and every third
//     keyframe of the CTA's range; the MMA warp and the producer interleave the three streams' tiles.  A (query,
//     keyframe) list therefore lives in ONE thread's registers from the first tile to the output — no cross-group
//     merge, no shared-memory lists, no CTA barrier per keyframe — and three tiles are in different phases at any time.
namespace xt {
constexpr int KX = 288;                       // operand bytes per row
constexpr int NSLICE = KX / 32;               // 9 instructions of K = 32 per tile
constexpr int TILE_BYTES = TN * KX;           // 36864
constexpr int XSTAGES = 5;                    // shared-memory ring (180 KB)
constexpr int NGRP = 3;                       // streams = epilogue groups = accumulators
constexpr int EPI_WARPS = 4 * NGRP;
constexpr int TMA_WARP = EPI_WARPS;
constexpr int MMA_WARP_X = EPI_WARPS + 1;
constexpr int XTHREADS = (MMA_WARP_X + 1) * 32;
constexpr uint32_t XA_COL = NGRP * 128;       // query operand: TMEM columns [384, 456)
constexpr int kKeyInvalid = 32896;            // keys >= this are "no row"
constexpr size_t kSmemBytes = (size_t)XSTAGES * TILE_BYTES + 1024;

__device__ __forceinline__ uint32_t xrow_off(int r) { return (uint32_t)(r >> 3) * (KX * 8) + (uint32_t)(r & 7) * 16; }

// ---- packed 256-bit rows (32 bytes) ----
// train side: a row is expanded by TWO threads (half = 0/1), 16 packed bytes each
__device__ __forceinline__ uint4 load_half(const uint8_t* __restrict__ row, int half) { return ldg_nc(row + 16 * half); }
// writes operand chunks 8 half .. 8 half + 7 of the row and returns the partial popcount
__device__ __forceinline__ int store_half(const uint4 v, int half, uint8_t* dst_row0) {
  const uint32_t w[4] = {v.x, v.y, v.z, v.w};
  int pc = 0;
#pragma unroll
  for (int i = 0; i < 4; i++) {
    pc += __popc(w[i]);
    // byte j of output word k is 0x80 (-128 as s8) if bit (k + 8 j) of w[i] is set, else 0; the query side uses the same
    // permutation with 0/2 bytes (tc_xt_kernel).  The left shift is a multiply so that it issues on the FMA pipe; only
    // the mask uses the (narrower) ALU pipe.
    uint4 lo, hi;
    lo.x = (w[i] * 128u) & 0x80808080u; lo.y = (w[i] * 64u) & 0x80808080u; lo.z = (w[i] * 32u) & 0x80808080u; lo.w = (w[i] * 16u) & 0x80808080u;
    hi.x = (w[i] * 8u) & 0x80808080u; hi.y = (w[i] * 4u) & 0x80808080u; hi.z = (w[i] * 2u) & 0x80808080u; hi.w = w[i] & 0x80808080u;
    *reinterpret_cast<uint4*>(dst_row0 + (8 * half + 2 * i) * 128) = lo;
    *reinterpret_cast<uint4*>(dst_row0 + (8 * half + 2 * i + 1) * 128) = hi;
  }
  return pc;
}
// query side (one thread per row): the 8 packed words and the row's popcount
__device__ __forceinline__ int load_q(const uint8_t* __restrict__ row, uint32_t (&w)[8]) {
  const uint4 a = ldg_nc(row), b = ldg_nc(row + 16);
  w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w; w[4] = b.x; w[5] = b.y; w[6] = b.z; w[7] = b.w;
  int pc = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) pc += __popc(w[i]);
  return pc;
}

// ---- one-time expansion (also the append path of the map database) ----
__global__ void __launch_bounds__(256) expand_tiles_kernel(const uint8_t* __restrict__ t, const int32_t* __restrict__ seg_ptr,
                                                           const int32_t* __restrict__ seg_tile, int seg_lo, int seg_hi,
                                                           int tile_lo, uint8_t* __restrict__ out) {
  const int tile = tile_lo + blockIdx.x;
  int lo = seg_lo, hi = seg_hi - 1;             // the last segment whose first tile is <= tile (skips empty segments)
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (seg_tile[mid] <= tile) lo = mid; else hi = mid - 1;
  }
  const int s_begin = seg_ptr[lo], len = seg_ptr[lo + 1] - s_begin, r0 = (tile - seg_tile[lo]) * TN;
  const int pt = threadIdx.x, prow = (pt & 7) | ((pt >> 4) << 3), half = (pt >> 3) & 1;
  const bool rv = r0 + prow < len;
  uint8_t* dst = out + (size_t)tile * TILE_BYTES + xrow_off(prow);
  int part = 0;
  if (rv) {
    part = store_half(load_half(t + (size_t)(s_begin + r0 + prow) * 32, half), half, dst);
  } else {
#pragma unroll
    for (int c = 0; c < 8; c++) *reinterpret_cast<uint4*>(dst + (8 * half + c) * 128) = make_uint4(0, 0, 0, 0);
  }
  part += __shfl_xor_sync(0xffffffffu, part, 8);
  if (half == 0) {
    uint4 key = make_uint4(0x7F7F7F7Fu, 0, 0, 0);
    if (rv) {
      const int p1 = min(part, 127), p2 = min(part - p1, 127), p3 = part - p1 - p2;
      key.x = (uint32_t)prow | ((uint32_t)p1 << 8) | ((uint32_t)p2 << 16) | ((uint32_t)p3 << 24);
      key.y = 0x00404040u;
    }
    *reinterpret_cast<uint4*>(dst + 16 * 128) = key;
  } else {
    *reinterpret_cast<uint4*>(dst + 17 * 128) = make_uint4(0, 0, 0, 0);
  }
}

// the interleaved tile sequence of a CTA: stream g walks keyframes seg0 + g, seg0 + g + NGRP, ... ; round-robin over the
// streams that still have tiles.  Producer, MMA warp and (per stream) the epilogue groups generate the same sequence.
struct Streams {
  int seg[NGRP], t[NGRP], nt[NGRP], tile0[NGRP];
  int seg1;
  const int32_t* seg_tile;
  __device__ void load(int g) {          // position stream g on its next non-empty keyframe (or past the end)
    while (seg[g] < seg1) {
      tile0[g] = seg_tile[seg[g]];
      nt[g] = seg_tile[seg[g] + 1] - tile0[g];
      if (nt[g] > 0) break;
      seg[g] += NGRP;
    }
    t[g] = 0;
  }
  __device__ void init(int seg0, int seg1_, const int32_t* st) {
    seg1 = seg1_; seg_tile = st;
#pragma unroll
    for (int g = 0; g < NGRP; g++) { seg[g] = seg0 + g; nt[g] = 0; tile0[g] = 0; load(g); }
  }
  __device__ bool active(int g) const { return seg[g] < seg1; }
  __device__ bool any() const { return seg[0] < seg1 || seg[1] < seg1 || seg[2] < seg1; }
  __device__ void advance(int g) {
    if (++t[g] >= nt[g]) { seg[g] += NGRP; load(g); }
  }
};

template <int K>
__global__ void __launch_bounds__(XTHREADS, 1) tc_xt_kernel(const TcParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* sB = smem;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)XSTAGES * TILE_BYTES);
  uint64_t* full = bars;                  // [XSTAGES] TMA bytes landed (expect_tx)
  uint64_t* empty = bars + XSTAGES;       // [XSTAGES] MMAs that read the stage completed (tcgen05.commit)
  uint64_t* tfull = bars + 2 * XSTAGES;   // [NGRP] accumulator g complete (tcgen05.commit)
  uint64_t* tempty = tfull + NGRP;        // [NGRP] accumulator g read back by its 4 warps
  __shared__ uint32_t tmem_base_s;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int qb = blockIdx.x % p.nqb, part = blockIdx.x / p.nqb;
  const int seg0 = (int)((long)part * p.n_seg / p.parts), seg1 = (int)((long)(part + 1) * p.n_seg / p.parts);

  if (tid == 0) {
    for (int s = 0; s < XSTAGES; s++) { cvb_mbar_init(&full[s], 1); cvb_mbar_init(&empty[s], 1); }
    for (int g = 0; g < NGRP; g++) { cvb_mbar_init(&tfull[g], 1); cvb_mbar_init(&tempty[g], 4); }
    cvb_fence_mbar_init();
  }
  if (warp == MMA_WARP_X) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(cvb_smem_addr(&tmem_base_s)));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;
  if (tid < TM) {
    // query block → tensor memory (thread = row = lane): data bytes 0/2, then the key slice
    const int q = qb * TM + tid;
    uint32_t w[8];
    int pq = 0;
    if (q < p.nq) {
      pq = load_q(p.q + (size_t)q * 32, w);
    } else {
#pragma unroll
      for (int i = 0; i < 8; i++) w[i] = 0;
    }
    const uint32_t a_taddr = tmem_base + ((uint32_t)(warp * 32) << 16) + XA_COL;
#pragma unroll
    for (int i = 0; i < 8; i++) {
      uint32_t r[8];
#pragma unroll
      for (int b = 0; b < 8; b++) r[b] = ((w[i] >> b) & 0x01010101u) * 2u;
      tc_st8(a_taddr + 8 * i, r);
    }
    {
      const int c4 = min(2 * pq, 255), c5 = min(2 * pq - c4, 255), c6 = 2 * pq - c4 - c5;
      uint32_t r[8] = {0, 0, 0, 0, 0, 0, 0, 0};
      if (q < p.nq) { r[0] = 0x80808001u; r[1] = (uint32_t)c4 | ((uint32_t)c5 << 8) | ((uint32_t)c6 << 16); }
      tc_st8(a_taddr + 64, r);
    }
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();

  if (warp == TMA_WARP) {
    // =================================== producer: one thread, bulk copies ===================================
    if (lane == 0) {
      Streams S;
      S.init(seg0, seg1, p.seg_tile);
      int n = 0;
      while (S.any()) {
#pragma unroll
        for (int g = 0; g < NGRP; g++) {
          if (!S.active(g)) continue;
          const int s = n % XSTAGES;
          if (n >= XSTAGES) cvb_mbar_wait(&empty[s], ((n / XSTAGES) - 1) & 1);
          cvb_mbar_expect_tx(&full[s], TILE_BYTES);
          const uint8_t* src = p.xt + (size_t)(S.tile0[g] + S.t[g]) * TILE_BYTES;
          uint8_t* dst = sB + (size_t)s * TILE_BYTES;
#pragma unroll
          for (int c = 0; c < 4; c++) cvb_bulk_g2s(dst + c * (TILE_BYTES / 4), src + c * (TILE_BYTES / 4), TILE_BYTES / 4, &full[s]);
          S.advance(g);
          n++;
        }
      }
    }
    __syncwarp();
  } else if (warp == MMA_WARP_X) {
    // =================================== MMA issuer (warp-uniform, one elected lane) ===================================
    // instruction descriptor: D = s32, A = u8, B = s8, both K-major, N = 128, M = 128
    const uint32_t idesc = (2u << 4) | (0u << 7) | (1u << 10) | ((uint32_t)(TN >> 3) << 17) | ((uint32_t)(TM >> 4) << 24);
    const uint32_t a_tmem = tmem_base + XA_COL;
    const uint32_t b_addr0 = cvb_smem_addr(sB);
    Streams S;
    S.init(seg0, seg1, p.seg_tile);
    int n = 0, j[NGRP] = {0, 0, 0};
    while (S.any()) {
#pragma unroll
      for (int g = 0; g < NGRP; g++) {
        if (!S.active(g)) continue;
        const int s = n % XSTAGES;
        cvb_mbar_wait(&full[s], (n / XSTAGES) & 1);
        if (j[g] >= 1) cvb_mbar_wait(&tempty[g], (j[g] - 1) & 1);
        tc_fence_after();
        const uint64_t b_desc0 = make_desc(b_addr0 + (uint32_t)s * TILE_BYTES, 128, KX * 8);
        const uint32_t d_tmem = tmem_base + (uint32_t)g * TN;
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < NSLICE; k++)
            tc_mma_i8_ts(d_tmem, a_tmem + 8 * k, b_desc0 + (uint64_t)(k * 16), idesc, k > 0 ? 1u : 0u);
          tc_commit(&empty[s]);
          tc_commit(&tfull[g]);
        }
        __syncwarp();
        S.advance(g);
        j[g]++;
        n++;
      }
    }
  } else {
    // =================================== epilogue group g: every NGRP-th keyframe, start to finish ===================================
    const int g = warp >> 2;
    const int row = (warp & 3) * 32 + lane;
    const int q = qb * TM + row;
    const bool valid = q < p.nq;
    const uint32_t taddr = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)g * TN;
    int jt = 0;
    for (int seg = seg0 + g; seg < seg1; seg += NGRP) {
      const int nt = p.seg_tile[seg + 1] - p.seg_tile[seg];
      int wk[K];   // (distance << kIdxBits) + row within the keyframe, ascending
#pragma unroll
      for (int c = 0; c < K; c++) wk[c] = INT_MAX;
      for (int t = 0; t < nt; t++, jt++) {
        cvb_mbar_wait(&tfull[g], jt & 1);
        tc_fence_after();
        uint32_t acc[64];
        tc_ld64_pack16(taddr, acc);            // 128 columns: register i = columns 2 i (low half) and 2 i + 1 (high half)
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tempty[g]);   // accumulator in registers: the MMA warp may start this stream's next tile
        if (valid) {
          unsigned pk[K];
#pragma unroll
          for (int c = 0; c < K; c++) pk[c] = 0xFFFFFFFFu;
#pragma unroll
          for (int i = 0; i < 64; i++) {
            unsigned x = acc[i];
#pragma unroll
            for (int c = 0; c < K; c++) {
              const unsigned lo = __vminu2(pk[c], x);
              x = __vmaxu2(pk[c], x);
              pk[c] = lo;
            }
          }
          // later tiles hold larger row indices: a candidate enters only with a strictly smaller distance than the k-th entry
          const unsigned best16 = min(pk[0] & 0xFFFFu, pk[0] >> 16);
          const int worst_d = wk[K - 1] == INT_MAX ? 1024 : (wk[K - 1] >> kIdxBits);
          if ((int)(best16 >> 7) < worst_d) {
#pragma unroll
            for (int c = 0; c < K; c++)
#pragma unroll
              for (int h = 0; h < 2; h++) {
                const unsigned k16 = h ? (pk[c] >> 16) : (pk[c] & 0xFFFFu);
                int x = k16 >= (unsigned)kKeyInvalid ? INT_MAX : (int)(((k16 >> 7) << kIdxBits) + (unsigned)(t * TN) + (k16 & 127u));
#pragma unroll
                for (int cc = 0; cc < K; cc++) {
                  const int lo = min(wk[cc], x);
                  x = max(wk[cc], x);
                  wk[cc] = lo;
                }
              }
          }
        }
      }
      // ---- keyframe finished: this thread holds the complete list of (query row, keyframe) ----
      int wi[K];
      float fd[K];
#pragma unroll
      for (int c = 0; c < K; c++) {
        wi[c] = wk[c] == INT_MAX ? -1 : (wk[c] & ((1 << kIdxBits) - 1));
        wk[c] = wk[c] == INT_MAX ? INT_MAX : (wk[c] >> kIdxBits);
        fd[c] = (float)wk[c];
      }
      if (p.filter) {
        bool ok = false;
        if (K >= 2 && valid) {
          const float dm = fd[0], dn = fd[K >= 2 ? 1 : 0];
          ok = wi[0] >= 0 && wi[K >= 2 ? 1 : 0] >= 0 && dm <= p.thr && dm < __fmul_rn(p.ratio, dn);
          const size_t o = (size_t)seg * p.nq + q;
          p.match_train[o] = ok ? wi[0] : -1;
          p.match_dist[o] = ok ? dm : FLT_MAX;
        }
        const unsigned b = __ballot_sync(0xffffffffu, ok);
        if (lane == 0 && b) atomicAdd(&p.n_matches[seg], __popc(b));
      } else if (valid) {
        const size_t o = ((size_t)seg * p.nq + q) * K;
#pragma unroll
        for (int c = 0; c < K; c++) {
          p.out_idx[o + c] = wi[c];
          reinterpret_cast<int32_t*>(p.out_dist)[o + c] = wi[c] >= 0 ? wk[c] : INT_MAX;
        }
      }
    }
  }
  // ---- teardown ----
  tc_fence_before();
  __syncthreads();
  if (warp == MMA_WARP_X) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base));
  }
}

template <int K>
int launch_xt(cvb_ctx* ctx, const TcParams& p, cudaStream_t st) {
  static cvb_once_per_device once;
  if (once.first(ctx->device)) {
    CVB_CUDA(ctx, cudaFuncSetAttribute(tc_xt_kernel<K>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBytes));
  }
  tc_xt_kernel<K><<<p.nqb * p.parts, XTHREADS, kSmemBytes, st>>>(p);
  CVB_CHECK_LAUNCH(ctx);
  return CVB_OK;
}
}  // namespace xt

int64_t tiles_of(const int32_t* h_seg, int n_seg, std::vector<int32_t>* seg_tile) {
  int64_t total = 0;
  if (seg_tile) seg_tile->assign((size_t)n_seg + 1, 0);
  for (int s = 0; s < n_seg; s++) {
    total += (h_seg[s + 1] - h_seg[s] + TN - 1) / TN;
    if (seg_tile) (*seg_tile)[s + 1] = (int32_t)total;
  }
  return total;
}
size_t tile_bytes() { return xt::TILE_BYTES; }

int expand_tiles(cvb_ctx* ctx, const uint8_t* d_rows, const int32_t* d_seg_ptr, const int32_t* d_seg_tile, int seg_lo, int seg_hi,
                 int tile_lo, int n_tiles, uint8_t* d_xt, cudaStream_t st) {
  if (n_tiles <= 0) return CVB_OK;
  xt::expand_tiles_kernel<<<n_tiles, 256, 0, st>>>(d_rows, d_seg_ptr, d_seg_tile, seg_lo, seg_hi, tile_lo, d_xt);
  CVB_CHECK_LAUNCH(ctx);
  return CVB_OK;
}

template <int K>
int launch_tc(cvb_ctx* ctx, const TcParams& p, cudaStream_t st) {
  static cvb_once_per_device once;
  const size_t smem = smem_bytes<K>();
  if (once.first(ctx->device)) {
    CVB_CUDA(ctx, cudaFuncSetAttribute(tc_scan_kernel<K>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  }
  tc_scan_kernel<K><<<p.nqb * p.parts, NUM_THREADS, smem, st>>>(p);
  CVB_CHECK_LAUNCH(ctx);
  return CVB_OK;
}

Formulation choose(const cvb_ctx* ctx, int nq, int n_seg, int64_t total_rows, int max_seg_len, bool filter) {
  const char* e = getenv("COVINS_B200_MATCH_KERNEL");
  const bool popc = e && !strcmp(e, "popc"), tc = e && !strcmp(e, "tc");
  const int nqb = (nq + TM - 1) / TM;
  const int parts = ctx->sm_count / nqb > 0 ? ctx->sm_count / nqb : 1;   // CTAs per query block that fill the GPU
  const bool big = (int64_t)nq * total_rows >= ((int64_t)1 << 26);
  // packed (distance, index) keys need < 4 Mi rows per segment
  if (max_seg_len < (1 << kIdxBits) && (tc ? (n_seg >= 1 && nq >= 1) : (!popc && n_seg >= parts && big))) return {Formulation::kPerSegment, 0};
  // one very long segment (map-wide k-NN): too few segments to spread over the SMs → about 4 uniform chunks per CTA, each
  // a multiple of TN and below the key's index range
  if (!filter && n_seg == 1 && !popc && big && total_rows >= (int64_t)parts * 4 * 1024) {
    const int64_t n_ps = parts * 4;
    const int64_t chunk = ((total_rows + n_ps - 1) / n_ps + TN - 1) / TN * TN;
    return {Formulation::kChunked, std::min(chunk, ((int64_t)1 << kIdxBits) - TN)};
  }
  return {Formulation::kScalar, 0};
}

int launch(cvb_ctx* ctx, TcParams p, int metric, int k, cudaStream_t st) {
  p.nqb = (p.nq + TM - 1) / TM;
  int parts = ctx->sm_count / p.nqb;
  if (parts < 1) parts = 1;
  if (parts > p.n_seg) parts = p.n_seg;
  p.parts = parts;
  if (metric == 0) {
    if (!p.xt) {
      // no resident tile store for this train set (raw-pointer API): expand it into the workspace first (HBM-bound pre-pass)
      CVB_REQUIRE(ctx, p.h_seg != nullptr, "tensor-core Hamming path needs the host copy of the segment table");
      std::vector<int32_t> h_tile;
      const int64_t n_tiles = tiles_of(p.h_seg, p.n_seg, &h_tile);
      int32_t* d_tile = (int32_t*)cvb_ws(ctx, WS_XT_TILE, sizeof(int32_t) * ((size_t)p.n_seg + 1));
      uint8_t* d_xt = (uint8_t*)cvb_ws(ctx, WS_XT, (size_t)n_tiles * xt::TILE_BYTES);
      if (!d_tile || !d_xt) return CVB_ERR_CUDA;
      CVB_CUDA(ctx, cudaMemcpyAsync(d_tile, h_tile.data(), sizeof(int32_t) * ((size_t)p.n_seg + 1), cudaMemcpyHostToDevice, st));
      CVB_CUDA(ctx, cudaStreamSynchronize(st));   // h_tile goes out of scope
      const int rc = expand_tiles(ctx, p.t, p.seg_ptr, d_tile, 0, p.n_seg, 0, (int)n_tiles, d_xt, st);
      if (rc) return rc;
      p.xt = d_xt;
      p.seg_tile = d_tile;
    }
    switch (k) {
      case 1: return xt::launch_xt<1>(ctx, p, st);
      case 2: return xt::launch_xt<2>(ctx, p, st);
      case 3: return xt::launch_xt<3>(ctx, p, st);
      default: return xt::launch_xt<4>(ctx, p, st);
    }
  }
  switch (k) {
    case 1: return launch_tc<1>(ctx, p, st);
    case 2: return launch_tc<2>(ctx, p, st);
    case 3: return launch_tc<3>(ctx, p, st);
    default: return launch_tc<4>(ctx, p, st);
  }
}

}  // namespace cvb_tc
