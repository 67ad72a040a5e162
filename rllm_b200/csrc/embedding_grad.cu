// Input-embedding term of a tied lm_head's gradient:  d_weight[id] += sum_{p : ids[p] = id} d_embeds[p]  (DESIGN.md section 4f).
//
// In a tied model the lm_head matrix is also the input embedding; the reference gets this term from autograd of the shared
// `embed_tokens` / `lm_head` parameter inside verl's actor update.  Here the order of every sum is fixed on the host
// (rllm_b200_token_segments: positions sorted stably by id, runs cut into pieces of at most RLLM_B200_SEGMENT_PIECE), so the
// fold has no atomics and every d_weight row has exactly one writer: bit-identical run to run, whatever the SM count.
//   pass 1  one warp per (piece, 256-column tile): sum the piece's rows in ascending position in fp32 registers (8 bf16 per lane,
//           16-byte loads), then add the sum to the d_weight row (a piece that is its whole segment) or store it as a partial
//   pass 2  one warp per (multi-piece segment, tile): add its partials in piece order, then add the sum to the row
// HBM-bound: n_in * H * 2 bytes read + n_distinct * H * 8 bytes (read-modify-write of the fp32 rows) + partials.
#include "common.cuh"

namespace rb {

constexpr int kEgThreads = 256;
constexpr int kEgTile = 256;  // columns per warp: 32 lanes x 8 bf16
constexpr int kEgUnroll = 4;  // rows in flight per lane

__device__ __forceinline__ void add_bf16x8(float (&acc)[8], const uint4 v) {
  acc[0] += bf16_lo(v.x);
  acc[1] += bf16_hi(v.x);
  acc[2] += bf16_lo(v.y);
  acc[3] += bf16_hi(v.y);
  acc[4] += bf16_lo(v.z);
  acc[5] += bf16_hi(v.z);
  acc[6] += bf16_lo(v.w);
  acc[7] += bf16_hi(v.w);
}

__device__ __forceinline__ void add_to_row(float* __restrict__ dst, const float (&acc)[8]) {
  float4* d4 = reinterpret_cast<float4*>(dst);
  float4 a = d4[0], b = d4[1];
  a.x += acc[0];
  a.y += acc[1];
  a.z += acc[2];
  a.w += acc[3];
  b.x += acc[4];
  b.y += acc[5];
  b.z += acc[6];
  b.w += acc[7];
  d4[0] = a;
  d4[1] = b;
}

__global__ void __launch_bounds__(kEgThreads) embedding_grad_pieces_kernel(const uint16_t* __restrict__ G, int64_t ldg, const int32_t* __restrict__ perm,
                                                                           const int32_t* __restrict__ piece_off, const int32_t* __restrict__ piece_row,
                                                                           const int32_t* __restrict__ piece_slot, int n_pieces, int n_tiles,
                                                                           float* __restrict__ partials, float* __restrict__ dW, int64_t lddw, int hidden, int vocab) {
  const int lane = threadIdx.x & 31;
  const int64_t n_items = static_cast<int64_t>(n_pieces) * n_tiles;
  const int64_t warps = static_cast<int64_t>(gridDim.x) * (kEgThreads / 32);
  for (int64_t item = (static_cast<int64_t>(blockIdx.x) * kEgThreads + threadIdx.x) >> 5; item < n_items; item += warps) {
    const int p = static_cast<int>(item / n_tiles);
    const int col = static_cast<int>(item - static_cast<int64_t>(p) * n_tiles) * kEgTile + lane * 8;
    const int row = __ldg(piece_row + p);
    if (col >= hidden || row < 0 || row >= vocab) continue;
    const int lo = __ldg(piece_off + p), hi = __ldg(piece_off + p + 1);
    float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    int j = lo;
    for (; j + kEgUnroll <= hi; j += kEgUnroll) {  // loads of kEgUnroll rows in flight, added in ascending position
      uint4 v[kEgUnroll];
#pragma unroll
      for (int u = 0; u < kEgUnroll; ++u) v[u] = __ldg(reinterpret_cast<const uint4*>(G + static_cast<int64_t>(__ldg(perm + j + u)) * ldg + col));
#pragma unroll
      for (int u = 0; u < kEgUnroll; ++u) add_bf16x8(acc, v[u]);
    }
    for (; j < hi; ++j) add_bf16x8(acc, __ldg(reinterpret_cast<const uint4*>(G + static_cast<int64_t>(__ldg(perm + j)) * ldg + col)));
    const int slot = __ldg(piece_slot + p);
    if (slot < 0) {
      add_to_row(dW + static_cast<int64_t>(row) * lddw + col, acc);
    } else {
      float4* d4 = reinterpret_cast<float4*>(partials + static_cast<int64_t>(slot) * hidden + col);
      d4[0] = make_float4(acc[0], acc[1], acc[2], acc[3]);
      d4[1] = make_float4(acc[4], acc[5], acc[6], acc[7]);
    }
  }
}

__global__ void __launch_bounds__(kEgThreads) embedding_grad_merge_kernel(const int32_t* __restrict__ multi_row, const int32_t* __restrict__ multi_slot_off, int n_multi,
                                                                          int n_tiles, const float* __restrict__ partials, float* __restrict__ dW, int64_t lddw, int hidden,
                                                                          int vocab) {
  const int lane = threadIdx.x & 31;
  const int64_t n_items = static_cast<int64_t>(n_multi) * n_tiles;
  const int64_t warps = static_cast<int64_t>(gridDim.x) * (kEgThreads / 32);
  for (int64_t item = (static_cast<int64_t>(blockIdx.x) * kEgThreads + threadIdx.x) >> 5; item < n_items; item += warps) {
    const int m = static_cast<int>(item / n_tiles);
    const int col = static_cast<int>(item - static_cast<int64_t>(m) * n_tiles) * kEgTile + lane * 8;
    const int row = __ldg(multi_row + m);
    if (col >= hidden || row < 0 || row >= vocab) continue;
    float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int s = __ldg(multi_slot_off + m), e = __ldg(multi_slot_off + m + 1); s < e; ++s) {
      const float4* p4 = reinterpret_cast<const float4*>(partials + static_cast<int64_t>(s) * hidden + col);
      const float4 a = __ldg(p4), b = __ldg(p4 + 1);
      acc[0] += a.x;
      acc[1] += a.y;
      acc[2] += a.z;
      acc[3] += a.w;
      acc[4] += b.x;
      acc[5] += b.y;
      acc[6] += b.z;
      acc[7] += b.w;
    }
    add_to_row(dW + static_cast<int64_t>(row) * lddw + col, acc);
  }
}

static int eg_grid(int64_t items, int sms) {
  const int64_t want = (items + kEgThreads / 32 - 1) / (kEgThreads / 32);
  return static_cast<int>(want < 1 ? 1 : (want < sms * 16 ? want : sms * 16));
}

}  // namespace rb

extern "C" int rllm_b200_embedding_grad_accumulate(const void* d_embeds_dev, int64_t ld_in, const int32_t* perm_dev, const int32_t* piece_off_dev,
                                                   const int32_t* piece_row_dev, const int32_t* piece_slot_dev, int32_t n_pieces, const int32_t* multi_row_dev,
                                                   const int32_t* multi_slot_off_dev, int32_t n_multi, float* partials_dev, float* d_weight_dev, int64_t lddw,
                                                   int32_t hidden, int32_t vocab, void* stream) {
  using namespace rb;
  RB_REQUIRE(n_pieces >= 0 && n_multi >= 0 && hidden > 0 && vocab > 0, "embedding_grad_accumulate: bad shape");
  if (n_pieces == 0) return 0;
  RB_REQUIRE(d_embeds_dev && perm_dev && piece_off_dev && piece_row_dev && piece_slot_dev && d_weight_dev, "embedding_grad_accumulate: NULL pointer");
  RB_REQUIRE(n_multi == 0 || (multi_row_dev && multi_slot_off_dev && partials_dev), "embedding_grad_accumulate: multi-piece segments need the merge tables and partials");
  RB_REQUIRE(hidden % 8 == 0 && ld_in % 8 == 0 && lddw % 4 == 0, "embedding_grad_accumulate: hidden and ld_in must be multiples of 8, lddw of 4");
  RB_REQUIRE(reinterpret_cast<uintptr_t>(d_embeds_dev) % 16 == 0 && reinterpret_cast<uintptr_t>(d_weight_dev) % 16 == 0 &&
                 reinterpret_cast<uintptr_t>(partials_dev) % 16 == 0,
             "embedding_grad_accumulate: operands must be 16-byte aligned");
  const int sms = sm_count();
  RB_REQUIRE(sms > 0, "embedding_grad_accumulate: no CUDA device");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int n_tiles = (hidden + kEgTile - 1) / kEgTile;
  embedding_grad_pieces_kernel<<<eg_grid(static_cast<int64_t>(n_pieces) * n_tiles, sms), kEgThreads, 0, st>>>(
      static_cast<const uint16_t*>(d_embeds_dev), ld_in, perm_dev, piece_off_dev, piece_row_dev, piece_slot_dev, n_pieces, n_tiles, partials_dev, d_weight_dev, lddw,
      hidden, vocab);
  RB_CUDA(cudaGetLastError());
  if (n_multi > 0) {
    embedding_grad_merge_kernel<<<eg_grid(static_cast<int64_t>(n_multi) * n_tiles, sms), kEgThreads, 0, st>>>(multi_row_dev, multi_slot_off_dev, n_multi, n_tiles,
                                                                                                              partials_dev, d_weight_dev, lddw, hidden, vocab);
    RB_CUDA(cudaGetLastError());
  }
  return 0;
}
