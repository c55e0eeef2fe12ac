// tc_match.cuh — interface of the tcgen05 (tensor-core) matching kernels, see tc_match.cu
#pragma once
#include <vector>

#include "cvb_internal.cuh"

namespace cvb_tc {

constexpr int kIdxBits = 22;   // Hamming packed key: distance << 22 | segment-local train index (segments < 4 Mi rows)

struct TcParams {
  const uint8_t* q;
  int nq;
  const uint8_t* t;
  const int32_t* seg_ptr;
  int n_seg;
  int nqb, parts;           // filled by launch()
  int32_t* out_idx;
  void* out_dist;
  int filter;
  float thr, ratio;
  int32_t* match_train;
  float* match_dist;
  int32_t* n_matches;
  // Hamming only: the pre-expanded operand tiles of the train set (expand_tiles) and the first tile of every segment
  // [n_seg + 1]; xt == nullptr → launch() expands into the workspace (needs h_seg, the host copy of seg_ptr)
  const uint8_t* xt;
  const int32_t* seg_tile;
  const int32_t* h_seg;
};

// metric 0 = Hamming (32-byte rows), 1 = L2 on u8 (128-byte rows); OpenCV k-NN rule (the DenseMatcher list rule is
// order dependent and stays on the scalar kernel)
int launch(cvb_ctx* ctx, TcParams p, int metric, int k, cudaStream_t st);

// Which formulation a k-NN request (nq >= 1) runs.  The tensor-core kernels are chosen when they fill the GPU: over the
// request's segments when there are enough of them, or — one very long segment, no fused filter — over uniform chunks of
// `chunk` rows whose lists the caller merges.  COVINS_B200_MATCH_KERNEL (read at every call): `popc` forces the scalar
// kernel, `tc` the per-segment tensor-core kernel wherever the packed keys can index the segments.
struct Formulation {
  enum Kind { kScalar, kPerSegment, kChunked } kind;
  int64_t chunk;   // kChunked only
};
Formulation choose(const cvb_ctx* ctx, int nq, int n_seg, int64_t total_rows, int max_seg_len, bool filter);

// pre-expanded operand store of the Hamming path: 128-row tiles per segment, tile_bytes() each
int64_t tiles_of(const int32_t* h_seg, int n_seg, std::vector<int32_t>* seg_tile);   // total tiles; optional prefix [n_seg + 1]
size_t tile_bytes();
int expand_tiles(cvb_ctx* ctx, const uint8_t* d_rows, const int32_t* d_seg_ptr, const int32_t* d_seg_tile, int seg_lo, int seg_hi,
                 int tile_lo, int n_tiles, uint8_t* d_xt, cudaStream_t st);

}  // namespace cvb_tc
