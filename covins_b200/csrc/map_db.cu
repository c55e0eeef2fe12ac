// map_db.cu — the merged map's ORB descriptors resident in HBM, queried per place-recognition request.
//
// Reference flow (covins_backend/src/covins_backend/placerec_gen_be.cpp:60-135): for every candidate keyframe the
// query keyframe's descriptor matrix is matched (knnMatch k=2 → distance + ratio filter) and only the accepted
// matches (img_matches, :102-114) and their count (:116-124) are consumed.  The descriptors of the map's keyframes
// never change after a keyframe is added (keyframe_be.cpp:106-137 fills them once from the message), so they are
// uploaded once (cvb_db_append) and stay in HBM; a query moves nq*32 B up and the accepted matches down.
#include <string.h>

#include <algorithm>

#include "cvb_internal.cuh"
#include "tc_match.cuh"

struct cvb_db {
  int desc_bytes = 32;
  uint8_t* d_rows = nullptr;
  size_t cap_rows = 0;
  std::vector<int32_t> seg_ptr{0};
  int32_t* d_seg = nullptr;
  size_t cap_seg = 0;
  bool seg_dirty = true;
  // the tensor-core matcher's operand tiles of every keyframe (tc_match.cu, "pre-expanded operand tiles"): written once
  // at append time, 128-row tiles, seg_tile[s] = first tile of keyframe s
  uint8_t* d_xt = nullptr;
  size_t cap_tiles = 0;
  std::vector<int32_t> seg_tile{0};
  int32_t* d_seg_tile = nullptr;
  // per-query scratch (grow-only)
  cvb_buf q, mt, md, nm, off, out_seg, out_q, out_t, out_d;
};

namespace {

int grow(cvb_ctx* ctx, cvb_buf& b, size_t bytes) {
  if (b.p && b.cap >= bytes) return CVB_OK;
  if (b.p) {
    CVB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    CVB_CUDA(ctx, cudaFree(b.p));
    b.p = nullptr;
    b.cap = 0;
  }
  const size_t want = std::max<size_t>(256, bytes + bytes / 4);
  CVB_CUDA(ctx, cudaMalloc(&b.p, want));
  b.cap = want;
  return CVB_OK;
}

// device copies of the segment tables
int refresh_seg(cvb_ctx* ctx, cvb_db* db) {
  if (!db->seg_dirty) return CVB_OK;
  cudaStream_t st = ctx->stream;
  if (db->cap_seg < db->seg_ptr.size()) {
    CVB_CUDA(ctx, cudaStreamSynchronize(st));
    if (db->d_seg) CVB_CUDA(ctx, cudaFree(db->d_seg));
    if (db->d_seg_tile) CVB_CUDA(ctx, cudaFree(db->d_seg_tile));
    db->d_seg = db->d_seg_tile = nullptr;
    db->cap_seg = db->seg_ptr.size() * 3 / 2 + 16;
    CVB_CUDA(ctx, cudaMalloc(&db->d_seg, db->cap_seg * sizeof(int32_t)));
    CVB_CUDA(ctx, cudaMalloc(&db->d_seg_tile, db->cap_seg * sizeof(int32_t)));
  }
  CVB_CUDA(ctx, cudaMemcpyAsync(db->d_seg, db->seg_ptr.data(), db->seg_ptr.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  CVB_CUDA(ctx, cudaMemcpyAsync(db->d_seg_tile, db->seg_tile.data(), db->seg_tile.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  CVB_CUDA(ctx, cudaStreamSynchronize(st));
  db->seg_dirty = false;
  return CVB_OK;
}

int reserve_tiles(cvb_ctx* ctx, cvb_db* db, size_t tiles, size_t used_tiles) {
  if (tiles <= db->cap_tiles) return CVB_OK;
  const size_t want = std::max(tiles, db->cap_tiles * 3 / 2), tb = cvb_tc::tile_bytes();
  uint8_t* p = nullptr;
  CVB_CUDA(ctx, cudaMalloc(&p, want * tb));
  const size_t used = used_tiles * tb;
  if (used) CVB_CUDA(ctx, cudaMemcpyAsync(p, db->d_xt, used, cudaMemcpyDeviceToDevice, ctx->stream));
  CVB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (db->d_xt) CVB_CUDA(ctx, cudaFree(db->d_xt));
  db->d_xt = p;
  db->cap_tiles = want;
  return CVB_OK;
}

// exclusive scan of the per-segment match counts; off[n_seg] = total.  One CTA, chunks of 1024 with a carry.
__global__ void __launch_bounds__(1024) db_offsets_kernel(const int32_t* __restrict__ cnt, int n_seg,
                                                           int32_t* __restrict__ off) {
  __shared__ int32_t warp_sum[32];
  __shared__ int32_t carry_s;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) carry_s = 0;
  __syncthreads();
  for (int base = 0; base < n_seg; base += 1024) {
    const int i = base + threadIdx.x;
    const int32_t v = i < n_seg ? cnt[i] : 0;
    int32_t x = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int32_t y = __shfl_up_sync(0xffffffffu, x, d);
      if (lane >= d) x += y;
    }
    if (lane == 31) warp_sum[warp] = x;
    __syncthreads();
    if (warp == 0) {
      int32_t w = warp_sum[lane];
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const int32_t y = __shfl_up_sync(0xffffffffu, w, d);
        if (lane >= d) w += y;
      }
      warp_sum[lane] = w;
    }
    __syncthreads();
    const int32_t carry = carry_s;
    const int32_t incl = x + (warp ? warp_sum[warp - 1] : 0) + carry;
    if (i < n_seg) off[i] = incl - v;
    __syncthreads();
    if (threadIdx.x == 1023) carry_s = incl;
    __syncthreads();
  }
  if (threadIdx.x == 0) off[n_seg] = carry_s;
}

// One warp per segment: accepted rows in query order (== the order of the reference's img_matches vector).
__global__ void __launch_bounds__(256) db_compact_kernel(const int32_t* __restrict__ mt, const float* __restrict__ md,
                                                          int nq, int n_seg, const int32_t* __restrict__ off, int cap,
                                                          int32_t* __restrict__ o_seg, int32_t* __restrict__ o_q,
                                                          int32_t* __restrict__ o_t, float* __restrict__ o_d) {
  const int seg = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (seg >= n_seg) return;
  const int lane = threadIdx.x & 31;
  int pos = off[seg];
  const int32_t* row_t = mt + (size_t)seg * nq;
  const float* row_d = md + (size_t)seg * nq;
  for (int q0 = 0; q0 < nq; q0 += 32) {
    const int q = q0 + lane;
    const int32_t t = q < nq ? row_t[q] : -1;
    const unsigned m = __ballot_sync(0xffffffffu, t >= 0);
    if (t >= 0) {
      const int p = pos + __popc(m & ((1u << lane) - 1u));
      if (p < cap) {
        o_seg[p] = seg;
        o_q[p] = q;
        o_t[p] = t;
        o_d[p] = row_d[q];
      }
    }
    pos += __popc(m);
  }
}

}  // namespace

extern "C" {

int cvb_db_create(cvb_ctx* ctx, int desc_bytes, cvb_db** out) {
  if (!ctx || !out) return CVB_ERR_INVALID;
  CVB_GUARD(ctx);
  *out = nullptr;
  if (desc_bytes != 32)
    return cvb_fail(ctx, CVB_ERR_UNSUPPORTED, "descriptor database: only 32-byte ORB descriptors, got %d", desc_bytes);
  cvb_db* db = new cvb_db();
  db->desc_bytes = desc_bytes;
  *out = db;
  return CVB_OK;
}

int cvb_db_destroy(cvb_ctx* ctx, cvb_db* db) {
  if (!db) return CVB_OK;
  if (ctx) cudaStreamSynchronize(ctx->stream);
  if (db->d_rows) cudaFree(db->d_rows);
  if (db->d_seg) cudaFree(db->d_seg);
  if (db->d_seg_tile) cudaFree(db->d_seg_tile);
  if (db->d_xt) cudaFree(db->d_xt);
  for (cvb_buf* b : {&db->q, &db->mt, &db->md, &db->nm, &db->off, &db->out_seg, &db->out_q, &db->out_t, &db->out_d})
    if (b->p) cudaFree(b->p);
  delete db;
  return CVB_OK;
}

int cvb_db_reserve(cvb_ctx* ctx, cvb_db* db, int64_t rows) {
  if (!ctx || !db || rows < 0) return CVB_ERR_INVALID;
  CVB_GUARD(ctx);
  if ((size_t)rows <= db->cap_rows) return CVB_OK;
  uint8_t* p = nullptr;
  CVB_CUDA(ctx, cudaMalloc(&p, (size_t)rows * db->desc_bytes));
  const size_t used = (size_t)db->seg_ptr.back() * db->desc_bytes;
  if (used) CVB_CUDA(ctx, cudaMemcpyAsync(p, db->d_rows, used, cudaMemcpyDeviceToDevice, ctx->stream));
  CVB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (db->d_rows) CVB_CUDA(ctx, cudaFree(db->d_rows));
  db->d_rows = p;
  db->cap_rows = (size_t)rows;
  return CVB_OK;
}

int cvb_db_append(cvb_ctx* ctx, cvb_db* db, const uint8_t* rows, const int32_t* rows_per_kf, int n_kf) {
  if (!ctx || !db) return CVB_ERR_INVALID;
  CVB_GUARD(ctx);
  CVB_REQUIRE(ctx, n_kf >= 0 && (n_kf == 0 || rows_per_kf), "cvb_db_append: bad arguments");
  int64_t add = 0;
  for (int i = 0; i < n_kf; ++i) {
    CVB_REQUIRE(ctx, rows_per_kf[i] >= 0, "cvb_db_append: negative row count");
    add += rows_per_kf[i];
  }
  const int64_t have = db->seg_ptr.back();
  CVB_REQUIRE(ctx, have + add < (int64_t)1 << 31, "cvb_db_append: more than 2^31 rows");
  CVB_REQUIRE(ctx, add == 0 || rows, "cvb_db_append: null rows");
  if ((size_t)(have + add) > db->cap_rows) {
    const int rc = cvb_db_reserve(ctx, db, std::max<int64_t>(have + add, (int64_t)(db->cap_rows * 3 / 2)));
    if (rc) return rc;
  }
  if (add) {
    CVB_CUDA(ctx, cudaMemcpyAsync(db->d_rows + (size_t)have * db->desc_bytes, rows, (size_t)add * db->desc_bytes,
                                  cudaMemcpyHostToDevice, ctx->stream));
    CVB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // `rows` may be freed by the caller on return
  }
  const int seg_old = (int)db->seg_ptr.size() - 1, tile_old = db->seg_tile.back();
  for (int i = 0; i < n_kf; ++i) {
    db->seg_ptr.push_back(db->seg_ptr.back() + rows_per_kf[i]);
    db->seg_tile.push_back(db->seg_tile.back() + (rows_per_kf[i] + 127) / 128);
  }
  db->seg_dirty = true;
  // the new keyframes' operand tiles (HBM-bound, once per keyframe; every later query reads them through the TMA engine)
  int rc = reserve_tiles(ctx, db, (size_t)db->seg_tile.back(), (size_t)tile_old);
  if (rc) return rc;
  if ((rc = refresh_seg(ctx, db))) return rc;
  rc = cvb_tc::expand_tiles(ctx, db->d_rows, db->d_seg, db->d_seg_tile, seg_old, seg_old + n_kf, tile_old,
                            db->seg_tile.back() - tile_old, db->d_xt, ctx->stream);
  if (rc) return rc;
  CVB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return CVB_OK;
}

int cvb_db_remove(cvb_ctx* ctx, cvb_db* db, int kf_index) {
  if (!ctx || !db) return CVB_ERR_INVALID;
  CVB_GUARD(ctx);
  const int n_seg = (int)db->seg_ptr.size() - 1;
  CVB_REQUIRE(ctx, kf_index >= 0 && kf_index < n_seg, "cvb_db_remove: keyframe index %d out of range (database holds %d)", kf_index, n_seg);
  const int64_t a = db->seg_ptr[kf_index], b = db->seg_ptr[kf_index + 1], end = db->seg_ptr.back();
  const size_t tail = (size_t)(end - b) * db->desc_bytes, len = (size_t)(b - a);
  if (tail && len) {   // move the tail down through a scratch buffer (source and destination overlap)
    void* tmp = cvb_ws(ctx, WS_GS2, tail);
    if (!tmp) return CVB_ERR_CUDA;
    CVB_CUDA(ctx, cudaMemcpyAsync(tmp, db->d_rows + (size_t)b * db->desc_bytes, tail, cudaMemcpyDeviceToDevice, ctx->stream));
    CVB_CUDA(ctx, cudaMemcpyAsync(db->d_rows + (size_t)a * db->desc_bytes, tmp, tail, cudaMemcpyDeviceToDevice, ctx->stream));
    CVB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  }
  {   // the same for the operand tiles
    const size_t tb = cvb_tc::tile_bytes();
    const int ta = db->seg_tile[kf_index], tbn = db->seg_tile[kf_index + 1], tend = db->seg_tile.back();
    const size_t ttail = (size_t)(tend - tbn) * tb;
    if (ttail && tbn > ta) {
      void* tmp = cvb_ws(ctx, WS_GS2, ttail);
      if (!tmp) return CVB_ERR_CUDA;
      CVB_CUDA(ctx, cudaMemcpyAsync(tmp, db->d_xt + (size_t)tbn * tb, ttail, cudaMemcpyDeviceToDevice, ctx->stream));
      CVB_CUDA(ctx, cudaMemcpyAsync(db->d_xt + (size_t)ta * tb, tmp, ttail, cudaMemcpyDeviceToDevice, ctx->stream));
      CVB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    db->seg_tile.erase(db->seg_tile.begin() + kf_index + 1);
    for (size_t i = (size_t)kf_index + 1; i < db->seg_tile.size(); i++) db->seg_tile[i] -= (int32_t)(tbn - ta);
  }
  db->seg_ptr.erase(db->seg_ptr.begin() + kf_index + 1);
  for (size_t i = (size_t)kf_index + 1; i < db->seg_ptr.size(); i++) db->seg_ptr[i] -= (int32_t)len;
  db->seg_dirty = true;
  return CVB_OK;
}

int cvb_db_size(const cvb_db* db, int32_t* n_kf, int64_t* n_rows) {
  if (!db) return CVB_ERR_INVALID;
  if (n_kf) *n_kf = (int32_t)db->seg_ptr.size() - 1;
  if (n_rows) *n_rows = db->seg_ptr.back();
  return CVB_OK;
}

int cvb_db_match_hamming_dev(cvb_ctx* ctx, cvb_db* db, const uint8_t* d_q, int nq, float thr, float ratio,
                             int32_t* d_match_train, float* d_match_dist, int32_t* d_n_matches, void* stream) {
  if (!ctx || !db) return CVB_ERR_INVALID;
  CVB_GUARD(ctx);
  const int n_seg = (int)db->seg_ptr.size() - 1;
  CVB_REQUIRE(ctx, nq >= 0 && (nq == 0 || d_q) && (n_seg == 0 || d_n_matches), "cvb_db_match_hamming_dev: bad arguments");
  if (n_seg == 0) return CVB_OK;
  int rc = refresh_seg(ctx, db);
  if (rc) return rc;
  return cvb_match_hamming_tiles_dev(ctx, d_q, nq, db->d_rows, db->d_seg, db->seg_ptr.data(), n_seg, thr, ratio, d_match_train,
                                     d_match_dist, d_n_matches, db->d_xt, db->d_seg_tile, cvb_stream(ctx, stream));
}

int cvb_db_match_hamming(cvb_ctx* ctx, cvb_db* db, const uint8_t* q, int nq, float thr, float ratio,
                         int32_t* n_matches, int32_t* m_kf, int32_t* m_query, int32_t* m_train, float* m_dist,
                         int cap, int32_t* n_total) {
  if (!ctx || !db) return CVB_ERR_INVALID;
  CVB_GUARD(ctx);
  const int n_seg = (int)db->seg_ptr.size() - 1;
  CVB_REQUIRE(ctx, nq >= 0 && cap >= 0 && n_total && (nq == 0 || q), "cvb_db_match_hamming: bad arguments");
  CVB_REQUIRE(ctx, cap == 0 || (m_kf && m_query && m_train && m_dist), "cvb_db_match_hamming: null outputs");
  *n_total = 0;
  if (n_seg == 0) return CVB_OK;
  if (nq == 0) {
    if (n_matches) std::fill(n_matches, n_matches + n_seg, 0);
    return CVB_OK;
  }
  cudaStream_t st = ctx->stream;
  int rc;
  if ((rc = refresh_seg(ctx, db))) return rc;
  const size_t on = (size_t)n_seg * nq;
  if ((rc = grow(ctx, db->q, (size_t)nq * 32))) return rc;
  if ((rc = grow(ctx, db->mt, on * 4))) return rc;
  if ((rc = grow(ctx, db->md, on * 4))) return rc;
  if ((rc = grow(ctx, db->nm, (size_t)n_seg * 4))) return rc;
  if ((rc = grow(ctx, db->off, (size_t)(n_seg + 1) * 4))) return rc;
  if (cap) {
    if ((rc = grow(ctx, db->out_seg, (size_t)cap * 4))) return rc;
    if ((rc = grow(ctx, db->out_q, (size_t)cap * 4))) return rc;
    if ((rc = grow(ctx, db->out_t, (size_t)cap * 4))) return rc;
    if ((rc = grow(ctx, db->out_d, (size_t)cap * 4))) return rc;
  }
  // pinned staging: [query | counts | offsets tail]
  const size_t pin_q = ((size_t)nq * 32 + 255) & ~(size_t)255;
  uint8_t* pin = (uint8_t*)cvb_pinned(ctx, pin_q + (size_t)(n_seg + 1) * 4 + 64);
  if (!pin) return CVB_ERR_CUDA;
  memcpy(pin, q, (size_t)nq * 32);
  CVB_CUDA(ctx, cudaMemcpyAsync(db->q.p, pin, (size_t)nq * 32, cudaMemcpyHostToDevice, st));
  rc = cvb_match_hamming_tiles_dev(ctx, (const uint8_t*)db->q.p, nq, db->d_rows, db->d_seg, db->seg_ptr.data(), n_seg, thr,
                                   ratio, (int32_t*)db->mt.p, (float*)db->md.p, (int32_t*)db->nm.p, db->d_xt, db->d_seg_tile, st);
  if (rc) return rc;
  db_offsets_kernel<<<1, 1024, 0, st>>>((const int32_t*)db->nm.p, n_seg, (int32_t*)db->off.p);
  CVB_CHECK_LAUNCH(ctx);
  if (cap) {
    db_compact_kernel<<<(n_seg + 7) / 8, 256, 0, st>>>((const int32_t*)db->mt.p, (const float*)db->md.p, nq, n_seg,
                                                       (const int32_t*)db->off.p, cap, (int32_t*)db->out_seg.p,
                                                       (int32_t*)db->out_q.p, (int32_t*)db->out_t.p,
                                                       (float*)db->out_d.p);
    CVB_CHECK_LAUNCH(ctx);
  }
  int32_t* pin_cnt = (int32_t*)(pin + pin_q);
  int32_t* pin_tot = pin_cnt + n_seg;
  CVB_CUDA(ctx, cudaMemcpyAsync(pin_cnt, db->nm.p, (size_t)n_seg * 4, cudaMemcpyDeviceToHost, st));
  CVB_CUDA(ctx, cudaMemcpyAsync(pin_tot, (int32_t*)db->off.p + n_seg, 4, cudaMemcpyDeviceToHost, st));
  CVB_CUDA(ctx, cudaStreamSynchronize(st));
  const int total = *pin_tot;
  *n_total = total;
  if (n_matches) memcpy(n_matches, pin_cnt, (size_t)n_seg * 4);
  const int n_out = std::min(total, cap);
  if (n_out) {
    CVB_CUDA(ctx, cudaMemcpyAsync(m_kf, db->out_seg.p, (size_t)n_out * 4, cudaMemcpyDeviceToHost, st));
    CVB_CUDA(ctx, cudaMemcpyAsync(m_query, db->out_q.p, (size_t)n_out * 4, cudaMemcpyDeviceToHost, st));
    CVB_CUDA(ctx, cudaMemcpyAsync(m_train, db->out_t.p, (size_t)n_out * 4, cudaMemcpyDeviceToHost, st));
    CVB_CUDA(ctx, cudaMemcpyAsync(m_dist, db->out_d.p, (size_t)n_out * 4, cudaMemcpyDeviceToHost, st));
    CVB_CUDA(ctx, cudaStreamSynchronize(st));
  }
  return CVB_OK;
}

}  // extern "C"
