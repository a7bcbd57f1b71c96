// train_common.cuh -- data layout shared by the training-mode forward (march_tc2_kernel<EMIT>) and the tensor-core
// backward (bwd_tc2.cuh): the tile plan, the per-tile activation / mask / gradient records and the mask bit order.
//
// The forward walks each CTA's rows in 128-row tiles (two per 256-row super-tile).  In training mode it leaves, per
// tile, a record of fp16 "tile images" -- [128 rows x C columns] in the shared-memory operand layout (K-blocks of 64
// columns, SWIZZLE_128B: row r of a K-block at (r>>3)*1024 + (r&7)*128, its 16-byte chunk c at ((c ^ (r&7)) << 4)), so
// that bulk copies make a tile MMA-ready again, as a K-major A operand (dgrad) or as an MN-major operand (wgrad:
// dW = dA^T H reduces over the sample rows).  In global memory an image is stored as TWO HALF IMAGES of 64 rows:
//   [half h = r >> 6][K-block kb = col >> 6][64 rows x 128 B = 8 KB]
// i.e. the 8 KB pieces of a K-block's upper and lower 64 rows are not adjacent (as they are in shared memory), the K-blocks of
// one 64-row half are: the weight gradient streams 64-row half tiles, and reads each operand as ONE contiguous C/64 x 8 KB
// piece instead of C/64 pieces 16 KB apart (HBM reads of scattered 8 KB pieces reach 4.1 TB/s, of 32 KB pieces 6.5: measured,
// profiles/r02_dram_stream_probe.jsonl).  A warp of the forward / dgrad epilogue owns 32 rows = a 4 KB slice of either layout.
//
//   activation record (forward -> backward), rec_act_bytes(D):
//     [0, 16 KB)                       enc    : gamma(p), 64 columns (63 + zero pad)
//     [16 KB + l * 64 KB), l < D       h_l    : post-ReLU output of pts_linears[l]        (run_nerf_helpers.py:99-101)
//     [16 KB + D * 64 KB), 32 KB       hv     : post-ReLU output of views_linears[0]       (:110-112)
//   (feature_linear's output is NOT recorded: its only consumer, the weight gradient of views_linears[0], is rewritten as
//    dW_v[:, :W] = (d_hv^T h_{D-1}) W_feat^T + db_v b_feat^T, which reads h_{D-1} -- already recorded -- instead)
//   mask record, rec_mask_bytes(D): sign bits of the pre-activations (1 = not positive = ReLU gradient 0)
//     layer l < D : l * 4096 + ch * 2048 + r * 16  : uint4 = columns [ch*128, ch*128+128), word b = columns b*32..
//     hv          : D * 4096 + ch * 1024 + r * 8   : uint2 = columns [ch*64, ch*64+64)
//     bit order inside a word: column (base + j) sits at bit (31 - j)   (built with one SHF.L.W per value)
//   gradient record (backward only), rec_grad_bytes(D): loss-scaled fp16 gradients w.r.t. PRE-activations
//     [0, 32 KB)                       d_hv   : seed, masked d(views pre-activation)
//     [32 KB + j * 64 KB), j = 0..D    step j output: j = 0 d_feat, j >= 1 dA_{D-j} (pre-activation of pts layer D-j)
#pragma once
#include "common.cuh"

namespace nb {

struct TilePlan {
  long long N; int S;
  int grid;            // CTAs of the forward launch (even: whole CTA pairs)
  int rays_per_cta;    // whole rays per CTA
  int nst;             // super-tiles (256 rows) per CTA: the record stride; a CTA may run fewer
  long long n_tiles;   // grid * nst * 2
};

// The forward's work split (launch_march): whole rays per CTA, balanced over the SMs, CTA pairs.
static inline TilePlan make_tile_plan(long long N, int S, int sms) {
  TilePlan t;
  t.N = N; t.S = S;
  const long long rows = N * (long long)S;
  const long long want = (rows + 255) / 256;
  int grid = (int)(want < sms ? want : sms);
  if (grid > N) grid = (int)N;
  if (grid < 1) grid = 1;
  t.rays_per_cta = (int)((N + grid - 1) / grid);
  grid = (int)((N + t.rays_per_cta - 1) / t.rays_per_cta);
  t.grid = (grid + 1) & ~1;
  t.nst = (int)(((long long)t.rays_per_cta * S + 255) / 256);
  t.n_tiles = (long long)t.grid * t.nst * 2;
  return t;
}

__host__ __device__ __forceinline__ uint32_t rec_act_bytes(int D) { return 16384u + (uint32_t)D * 65536u + 32768u; }
__host__ __device__ __forceinline__ uint32_t rec_act_h(int l) { return 16384u + (uint32_t)l * 65536u; }              // l < D
__host__ __device__ __forceinline__ uint32_t rec_act_hv(int D) { return 16384u + (uint32_t)D * 65536u; }
__host__ __device__ __forceinline__ uint32_t rec_mask_bytes(int D) { return (uint32_t)D * 4096u + 2048u; }
__host__ __device__ __forceinline__ uint32_t rec_grad_bytes(int D) { return 32768u + (uint32_t)(D + 1) * 65536u; }
__host__ __device__ __forceinline__ uint32_t rec_grad_step(int j) { return 32768u + (uint32_t)j * 65536u; }         // output of dgrad step j
__host__ __device__ __forceinline__ uint32_t rec_grad_dA(int l, int D) { return rec_grad_step(D - l); }              // pts layer l

// byte offset of element (row r, column col) inside a [128 x C] tile image in global memory
__host__ __device__ __forceinline__ uint32_t img_off(int r, int col, int C) {
  return (uint32_t)((r >> 6) * (C >> 6) * 8192 + (col >> 6) * 8192 + ((r & 63) >> 3) * 1024 + (r & 7) * 128 + ((((col & 63) >> 3) ^ (r & 7)) << 4) + (col & 7) * 2);
}
// byte offset of the 4 KB slice (rows 32 q .. 32 q + 31) of K-block kb inside a [128 x C] tile image in global memory
__host__ __device__ __forceinline__ uint32_t img_slice_off(int q, int kb, int C) {
  return (uint32_t)((q >> 1) * (C >> 6) * 8192 + kb * 8192 + (q & 1) * 4096);
}

// rows of CTA `cta` and the super-tiles its PAIR runs (both CTAs of a pair run the same number)
__host__ __device__ __forceinline__ int plan_cta_rows(long long N, int S, int rays_per_cta, int cta) {
  const long long r0 = (long long)cta * rays_per_cta;
  const long long r1 = (r0 + rays_per_cta < N) ? r0 + rays_per_cta : N;
  return (r1 > r0) ? (int)(r1 - r0) * S : 0;
}
__host__ __device__ __forceinline__ int plan_cta_nst(long long N, int S, int rays_per_cta, int cta) {
  const int a = plan_cta_rows(N, S, rays_per_cta, cta), b = plan_cta_rows(N, S, rays_per_cta, cta ^ 1);
  return ((a > b ? a : b) + 255) / 256;
}

// ---- mask bits ------------------------------------------------------------------------------------------------
// m = (m << 1) | sign(x): after 32 calls in column order, column j of the batch sits at bit (31 - j)
__device__ __forceinline__ uint32_t mask_push(uint32_t m, float x) { return __funnelshift_l(__float_as_uint(x), m, 1); }
// zero x when bit (31 - j) of m is set
__device__ __forceinline__ float mask_apply(uint32_t m, int j, float x) {
  const int t = ((int)(m << j)) >> 31;
  return __uint_as_float(__float_as_uint(x) & ~(uint32_t)t);
}

// static loss scale of the fp16 backward: a power of two that puts max |dL/drgb_map| at ~2^11
// (tools/bwd_precision_study.py: with the range handled, fp16 gradient operands cost nothing measurable)
__device__ __forceinline__ float loss_scale_from_absmax(float amax) {
  if (!(amax > 0.f) || !(amax < 3.0e38f)) return 1.0f;
  return exp2f(floorf(log2f(2048.0f / amax)));
}

}  // namespace nb
