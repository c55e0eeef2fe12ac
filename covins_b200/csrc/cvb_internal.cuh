// cvb_internal.cuh — ctx, error plumbing and small device helpers shared by all translation units of
// libcovins_b200.so.  Not part of the public boundary (that is include/covins_b200.h).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <atomic>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/covins_b200.h"

struct cvb_buf {
  void* p = nullptr;
  size_t cap = 0;
};

enum { WS_Q = 0, WS_T, WS_SEG, WS_OUT0, WS_OUT1, WS_OUT2, WS_PART_I, WS_PART_D, WS_LIST_I, WS_LIST_D, WS_SKIPA,
       WS_SKIPB, WS_TMP0, WS_TMP1, WS_FLAG, WS_MISC, WS_CHUNK_PS, WS_CHUNK_OFF, WS_GS0, WS_GS1, WS_GS2, WS_GS3, WS_GS4, WS_GS5, WS_XT, WS_XT_TILE,
       WS_COUNT };

struct cvb_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  int sm_count = 148;
  int64_t launches = 0;
  std::string err;
  // grow-only device workspaces (named slots so independent stages never alias)
  cvb_buf ws[WS_COUNT];
  // pinned host staging
  void* h_pin = nullptr;
  size_t h_pin_cap = 0;
  void* ba = nullptr;  // BA state (owned by ba_*.cu)
  // every extern "C" entry point holds this lock for its duration (cvb_device_guard): a ctx may be shared between host
  // threads — calls on one ctx are serialised, concurrency comes from one ctx per thread
  mutable std::recursive_mutex mtx;
};

// cudaFuncSetAttribute applies to the CURRENT device: one flag per (call site, device), so that a process that opens contexts
// on several GPUs raises the dynamic shared-memory limit on each of them
struct cvb_once_per_device {
  std::atomic<bool> done[64];
  cvb_once_per_device() { for (auto& d : done) d.store(false); }
  bool first(int device) {
    if (device < 0 || device >= 64) return true;
    return !done[device].exchange(true);
  }
};

int cvb_fail(cvb_ctx* ctx, int code, const char* fmt, ...);
void* cvb_ws(cvb_ctx* ctx, int slot, size_t bytes);          // returns nullptr on failure (ctx->err set)
void* cvb_pinned(cvb_ctx* ctx, size_t bytes);

// cvb_match_hamming_batch_dev without the entry-point guard (the caller holds it), with the train rows' resident operand
// tiles when there are any (xt / seg_tile as cvb_tc::TcParams; both null: the tensor-core path expands them per call)
int cvb_match_hamming_tiles_dev(cvb_ctx* ctx, const uint8_t* d_q, int nq, const uint8_t* d_t, const int32_t* d_seg_ptr,
                                const int32_t* h_seg_ptr, int n_seg, float thr, float ratio, int32_t* d_match_train,
                                float* d_match_dist, int32_t* d_n_matches, const uint8_t* xt, const int32_t* seg_tile,
                                cudaStream_t st);

#define CVB_CUDA(ctx, call)                                                                         \
  do {                                                                                              \
    cudaError_t e_ = (call);                                                                        \
    if (e_ != cudaSuccess)                                                                          \
      return cvb_fail((ctx), CVB_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_),  \
                      __FILE__, __LINE__);                                                          \
  } while (0)

#define CVB_CHECK_LAUNCH(ctx)                                                                       \
  do {                                                                                              \
    (ctx)->launches++;                                                                              \
    cudaError_t e_ = cudaGetLastError();                                                            \
    if (e_ != cudaSuccess)                                                                          \
      return cvb_fail((ctx), CVB_ERR_CUDA, "kernel launch failed: %s (%s:%d)",                      \
                      cudaGetErrorString(e_), __FILE__, __LINE__);                                  \
  } while (0)

#define CVB_REQUIRE(ctx, cond, ...)                                      \
  do {                                                                   \
    if (!(cond)) return cvb_fail((ctx), CVB_ERR_INVALID, __VA_ARGS__);   \
  } while (0)

static inline cudaStream_t cvb_stream(cvb_ctx* ctx, void* s) { return s ? (cudaStream_t)s : ctx->stream; }

// Scoped guard of every extern "C" entry point: takes the ctx's lock (calls on one ctx are serialised, so a ctx may be
// shared between host threads) and makes the ctx's device current for the calling thread (a new host thread defaults to
// device 0; two ctxs on different GPUs may be driven from one thread), restoring the previous device on exit.
struct cvb_device_guard {
  int prev = -1;
  bool switched = false;
  const cvb_ctx* ctx = nullptr;
  explicit cvb_device_guard(const cvb_ctx* c) : ctx(c) {
    if (c) c->mtx.lock();
    if (c && cudaGetDevice(&prev) == cudaSuccess && prev != c->device) switched = cudaSetDevice(c->device) == cudaSuccess;
  }
  ~cvb_device_guard() {
    if (switched) cudaSetDevice(prev);
    if (ctx) ctx->mtx.unlock();
  }
  cvb_device_guard(const cvb_device_guard&) = delete;
  cvb_device_guard& operator=(const cvb_device_guard&) = delete;
};
#define CVB_GUARD(ctx) cvb_device_guard cvb_guard_((ctx))

// ---------------------------------------------------------------------------------------------
// Device helpers: mbarrier + 1-D bulk TMA (cp.async.bulk → SASS UBLKCP), used to stage descriptor
// tiles into shared memory.
// ---------------------------------------------------------------------------------------------
#ifdef __CUDACC__
__device__ __forceinline__ uint32_t cvb_smem_addr(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void cvb_mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(cvb_smem_addr(bar)), "r"(count));
}
__device__ __forceinline__ void cvb_fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void cvb_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(cvb_smem_addr(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void cvb_mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE;\n"
      "bra WAIT_LOOP;\n"
      "DONE:\n"
      "}\n" ::"r"(cvb_smem_addr(bar)),
      "r"(parity)
      : "memory");
}
// global → shared bulk copy (bytes % 16 == 0, both addresses 16-B aligned), completion on `bar`.
__device__ __forceinline__ void cvb_bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          cvb_smem_addr(smem_dst)),
      "l"(gmem_src), "r"(bytes), "r"(cvb_smem_addr(bar))
      : "memory");
}
#endif
