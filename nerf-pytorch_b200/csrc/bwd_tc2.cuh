// bwd_tc2.cuh -- tensor-core backward of one network pass (row a11: loss.backward() through run_nerf.py:381-386 /
// :397-403, i.e. autograd's backward of NeRF.forward run_nerf_helpers.py:96-119 and raw2outputs run_nerf.py:262-305).
//
// Inputs: the per-tile records the training-mode forward left (train_common.cuh: fp16 activation images + ReLU sign
// masks), its raw [N,S,4] output, and dL/drgb_map.  Everything below works on 128-row tiles in the forward's own tile
// order, with activation gradients as loss-scaled fp16 (one power-of-two scale per pass taken from max |dL/drgb_map|,
// saturating conversions) and fp32 accumulation in TMEM:
//
//   raw2outputs_bwd_kernel (small_kernels.cuh)  dL/draw per sample                       (SURVEY App. E)
//   dhv_seed_heads_kernel  d_hv = relu'(hv) * (d_rgb W_rgb) as tile images + rgb_linear's weight / bias gradient (:114)
//   dgrad_tc2_kernel     the chain  d_hv -> d_feat -> dA_{D-1} -> ... -> dA_0  as tcgen05 cta_group::2 passes with
//                        TRANSPOSED weight chunks streamed through the forward's 7 x 8 KB TMA ring; the epilogue applies
//                        the ReLU mask (and the alpha_linear rank-1 term), writes the next A tile in place and the same
//                        tile goes to the gradient record, one 16 KB K-block per bulk store.  Same warp roles / barriers as the
//                        forward pair kernel (fused_tc2.cuh); activation gradients never leave the SM between layers.
//   wgrad_tc_kernel      dW_l += dA_l^T H_{l-1}: both operands MN-major straight from the images (no re-layout), the
//                        CTAs are partitioned over the layers so that each holds ONE layer's dW in TMEM across all of
//                        its tiles (256 x 256 fp32 = all 512 columns) and leaves the SM once; bias gradients are the
//                        column sums of the dA tiles while they sit in shared memory.
//   wgrad_reduce_kernel  sums the per-CTA partial dW, un-scales, adds into the gradient tensors
//                        (alpha_linear's gradient and the per-ray row sums of d_hv are computed by the wgrad kernel's spare
//                        warps from the tiles it streams anyway)
//   views_enc_wgrad_kernel  views_linears[0].weight[:, W:] from the per-ray sums and gamma(viewdir)
//   views_feat_wgrad_kernel views_linears[0].weight[:, :W] = (d_hv^T h_{D-1}) W_feat^T + db_v b_feat^T (feature_linear's output is never stored)
//
// TMEM capacity is what shapes this: one layer's dW fills an SM's tensor memory, so the weight gradient cannot share
// a kernel with a tile-major dgrad chain (ten layers would need ten SMs' worth); hence dgrad is tile-major (on-chip
// chain) and wgrad layer-major (streams the images once: 2 x 64 KB per tile-layer at 64 MAC/B -- HBM-bound).
#pragma once
#include <cuda.h>
#include "fused_tc.cuh"
#include "fused_tc2.cuh"
#include "train_common.cuh"

namespace nb {

// ---------------------------------------------------------------------------------------------------------------
// backward weight stream: step 0 = views_linears[0].weight[:, :W]^T (K = W/2: 4 chunks), step 1 = feature_linear^T,
// step j >= 2 = pts_linears[D+1-j].weight[:, h columns]^T (8 chunks each); every chunk is [N = 256 x K = 32] fp16 in the
// forward's SWIZZLE_64B K-major image, rank-split like the forward stream (pack_weights)
// ---------------------------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ int bwd_step_units(int j) { return j == 0 ? 4 : 8; }
static inline int bwd_stream_chunks(int D) { return 4 + 8 * D; }

// ---------------------------------------------------------------------------------------------------------------
// max |g| over n floats -> *out (bit pattern; non-negative floats order like unsigned ints).  *out zeroed by the caller.
// ---------------------------------------------------------------------------------------------------------------
__global__ void absmax_kernel(const float* __restrict__ g, long long n, unsigned int* __restrict__ out) {
  float m = 0.f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float v = fabsf(g[i]);
    m = (v > m || v != v) ? v : m;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { const float t = __shfl_xor_sync(0xffffffffu, m, o); m = (t > m || t != t) ? t : m; }
  if ((threadIdx.x & 31) == 0) atomicMax(out, __float_as_uint(m));
}

// gamma(viewdir) per ray (run_nerf.py:44-46 re-encodes it per sample): out [N, ICV]
__global__ void encv_kernel(const float* __restrict__ dirs, int stride, long long N, int ICV, float* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N * ICV) return;
  const long long n = i / ICV;
  const int c = (int)(i - n * ICV);
  const float* d = dirs + n * stride;
  float v;
  if (c < 3) v = d[c];
  else { const int f = (c - 3) / 6, q = (c - 3) % 6; const float a = __fmul_rn(d[q % 3], exp2f((float)f)); v = (q < 3) ? sinf(a) : cosf(a); }
  out[i] = v;
}

// ---------------------------------------------------------------------------------------------------------------
// rgb_linear's backward (run_nerf_helpers.py:114), both halves in one sweep over the rows:
//   seed of the dgrad chain: d_hv[row][c] = scale * (hv[row][c] > 0) * sum_j d_rgb[row][j] W_rgb[j][c]   (c < 128), written as the
//     first 32 KB of every tile's gradient record (rows beyond the CTA's range: zeros -- dgrad and wgrad rely on that);
//   weight / bias gradient: dW_rgb[j][c] += sum_rows d_rgb[row][j] hv[row][c],  db_rgb[j] += sum_rows d_rgb[row][j]   (fp32)
// One warp per row, lane = four columns: a row is 256 contiguous bytes of hv in and of d_hv out (two 128-byte lines each).
// ---------------------------------------------------------------------------------------------------------------
struct SeedParams {
  const float* d_raw; const uint8_t* mask; const uint8_t* act; uint8_t* grad; const float* rgb_w; const unsigned int* amax;
  long long N; int S, rays_per_cta, nst_plan, D;
  uint32_t rec_mask, rec_act, rec_grad; long long n_tiles;
  float* g_rgb_w; float* g_rgb_b;
};

__global__ void __launch_bounds__(256, 3) dhv_seed_heads_kernel(const SeedParams p) {
  __shared__ float s_acc[8][12 * 32 + 3];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int c = lane * 4, ch = lane >> 4, wsel = (lane >> 3) & 1, bit0 = c & 31;
  const float scale = loss_scale_from_absmax(__uint_as_float(*p.amax));
  float wr[4], wg[4], wb[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) { wr[i] = p.rgb_w[c + i] * scale; wg[i] = p.rgb_w[128 + c + i] * scale; wb[i] = p.rgb_w[256 + c + i] * scale; }
  float a[12];
#pragma unroll
  for (int i = 0; i < 12; ++i) a[i] = 0.f;
  float b0 = 0.f, b1 = 0.f, b2 = 0.f;
  for (long long t = blockIdx.x; t < p.n_tiles; t += gridDim.x) {
    const int cta = (int)(t / (2 * p.nst_plan)), st = (int)((t >> 1) % p.nst_plan), X = (int)(t & 1);
    if (st >= plan_cta_nst(p.N, p.S, p.rays_per_cta, cta)) continue;          // never read (neither CTA of the pair has rows there)
    const int nrows = plan_cta_rows(p.N, p.S, p.rays_per_cta, cta);
    const int lr0 = st * 256 + X * 128;
    const long long row_begin = (long long)cta * p.rays_per_cta * p.S;
    const int nv = (nrows - lr0 < 128) ? nrows - lr0 : 128;                   // (<= 0: the partner's rows only -> a tile of zeros)
    const uint8_t* hv = p.act + (size_t)t * p.rec_act + rec_act_hv(p.D);
    const uint8_t* mrec = p.mask + (size_t)t * p.rec_mask + (uint32_t)p.D * 4096u + (uint32_t)ch * 1024u + (uint32_t)wsel * 4u;
    uint8_t* const g = p.grad + (size_t)t * p.rec_grad;
    // warp w takes rows 16 w .. 16 w + 15: their dL/draw rows come in as ONE coalesced load (lane i < 16 holds row i's float4 and
    // hands it out by shuffle), which leaves the registers for all 16 hv / mask loads to be in flight at once (load-latency bound)
    const int rbase = warp * 16;
    float4 dmine = make_float4(0.f, 0.f, 0.f, 0.f);
    if (lane < 16 && rbase + lane < nv) dmine = reinterpret_cast<const float4*>(p.d_raw)[row_begin + lr0 + rbase + lane];
    uint2 hw[16];
    uint32_t mw[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      const int r = rbase + k;
      hw[k] = make_uint2(0u, 0u); mw[k] = 0u;
      if (r < nv) {
        hw[k] = *reinterpret_cast<const uint2*>(hv + img_off(r, c, 128));
        mw[k] = *reinterpret_cast<const uint32_t*>(mrec + (uint32_t)r * 8u);
      }
    }
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      const int r = rbase + k;
      const float dx = __shfl_sync(0xffffffffu, dmine.x, k), dy = __shfl_sync(0xffffffffu, dmine.y, k), dz = __shfl_sync(0xffffffffu, dmine.z, k);
      uint2 out = make_uint2(0u, 0u);
      if (r < nv) {
        const __half2 h01 = *reinterpret_cast<const __half2*>(&hw[k].x), h23 = *reinterpret_cast<const __half2*>(&hw[k].y);
        const float h[4] = {__low2float(h01), __high2float(h01), __low2float(h23), __high2float(h23)};
        float x[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          a[i] = fmaf(dx, h[i], a[i]); a[4 + i] = fmaf(dy, h[i], a[4 + i]); a[8 + i] = fmaf(dz, h[i], a[8 + i]);
          x[i] = mask_apply(mw[k], bit0 + i, fmaf(dx, wr[i], fmaf(dy, wg[i], dz * wb[i])));
        }
        b0 += dx; b1 += dy; b2 += dz;
        out = make_uint2(ptx::cvt_sat_f16x2(x[0], x[1]), ptx::cvt_sat_f16x2(x[2], x[3]));
      }
      *reinterpret_cast<uint2*>(g + img_off(r, c, 128)) = out;
    }
  }
#pragma unroll
  for (int i = 0; i < 12; ++i) s_acc[warp][i * 32 + lane] = a[i];
  if (lane == 0) { s_acc[warp][384] = b0; s_acc[warp][385] = b1; s_acc[warp][386] = b2; }
  __syncthreads();
  for (int i = threadIdx.x; i < 387; i += 256) {
    float v = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) v += s_acc[w][i];
    if (i < 384) {                                      // i = (j * 4 + k) * 32 + lane  ->  weight[j][lane * 4 + k]
      const int j = i / 128, k = (i / 32) & 3, ln = i & 31;
      atomicAdd(p.g_rgb_w + j * 128 + ln * 4 + k, v);
    } else atomicAdd(p.g_rgb_b + (i - 384), v);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// dgrad chain (CTA pair, cta_group::2) -- structure, warp roles and barrier protocol of march_tc2_kernel
// ---------------------------------------------------------------------------------------------------------------
struct DgradParams {
  const uint8_t* mask; uint8_t* grad; const float* d_raw; const unsigned int* amax; const float* alpha_w;
  long long N; int S, rays_per_cta, nst_plan, D;
  uint32_t rec_mask, rec_grad;
  unsigned long long pair_half_bytes;       // bytes of one rank's half of the backward chunk stream
};

constexpr uint32_t DG2_SEED = SM_ENC;                                        // 131072: 32 KB, d_hv of ONE slot
constexpr uint32_t DG2_ALPHA = SM_WRING + TC2_NST * TC2_STAGE_BYTES;         // 221184: alpha_linear.weight, 1 KB fp32
constexpr uint32_t DG2_BARS = DG2_ALPHA + 1024;                              // 222208
constexpr uint32_t DG2_MISC = DG2_BARS + 256;                                // 222464: tmem pointer
constexpr uint32_t DG2_TOTAL = DG2_MISC + 64;
static_assert(DG2_TOTAL <= SM_ALLOC, "dgrad shared-memory map exceeds the allocation");

// x[32] (one row, 32 consecutive columns starting at COL0 of this warp's column half) -> saturating fp16 -> four 16-byte
// stores into the swizzled A tile (sw[] as in store_act32_pre)
template <int COL0>
__device__ __forceinline__ void store_grad32_pre(const float (&x)[32], const uint32_t (&sw)[8]) {
  constexpr uint32_t kb = (uint32_t)(COL0 >> 6) * 16384u;
  constexpr int c16_0 = (COL0 & 63) >> 3;
#pragma unroll
  for (int g = 0; g < 4; ++g)
    ptx::st_shared_v4(sw[c16_0 + g] + kb, ptx::cvt_sat_f16x2(x[g * 8 + 0], x[g * 8 + 1]), ptx::cvt_sat_f16x2(x[g * 8 + 2], x[g * 8 + 3]),
                      ptx::cvt_sat_f16x2(x[g * 8 + 4], x[g * 8 + 5]), ptx::cvt_sat_f16x2(x[g * 8 + 6], x[g * 8 + 7]));
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(TC_THREADS, 1)
dgrad_tc2_kernel(const DgradParams p, const __grid_constant__ CUtensorMap wmap, const __grid_constant__ CUtensorMap gmap) {
  uint8_t* smem = tc_smem;
  const uint32_t sb = ptx::smem_u32(smem);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if ((sb & 1023u) != 0) __trap();
  const uint32_t rank = ptx::cluster_ctarank();
  const bool leader = (rank == 0);

  float* s_alpha = reinterpret_cast<float*>(smem + DG2_ALPHA);
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(smem + DG2_MISC);
  const uint32_t a_alpha = sb + DG2_ALPHA;
  const uint32_t bar_wfull = sb + DG2_BARS;            // [7] (leader): TMA bytes of both CTAs
  const uint32_t bar_wempty = sb + DG2_BARS + 56;      // [7] multicast commit
  const uint32_t bar_dfull = sb + DG2_BARS + 112;      // [2] multicast commit
  const uint32_t bar_act = sb + DG2_BARS + 128;        // [2] (leader) 16 epilogue warps
  const uint32_t bar_seedfull = sb + DG2_BARS + 144;   //     (leader) TMA bytes of both CTAs' seed tiles
  const uint32_t bar_seedfree = sb + DG2_BARS + 152;   //     multicast commit after the last step-0 MMA
  auto arrive_leader = [&](uint32_t bar) {
    __syncwarp();
    if (lane == 0) {
      if (leader) ptx::mbar_arrive(bar);
      else ptx::mbar_arrive_remote(ptx::mapa(bar, 0));
    }
  };

  // rows: exactly the forward's split -- the launch has the forward's grid, and CTA vc serves forward CTA vc (same rays, same
  // tile records)
  const int vc = (int)blockIdx.x;
  const int D = p.D, NS = D + 1, nst = plan_cta_nst(p.N, p.S, p.rays_per_cta, vc);

  for (int i = threadIdx.x; i < 256; i += TC_THREADS) s_alpha[i] = p.alpha_w[i];
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < TC2_NST; ++i) { ptx::mbar_init(bar_wfull + 8 * i, 1); ptx::mbar_init(bar_wempty + 8 * i, 1); }
    for (int x = 0; x < 2; ++x) {
      ptx::mbar_init(bar_dfull + 8 * x, 1); ptx::mbar_init(bar_act + 8 * x, 16);
    }
    ptx::mbar_init(bar_seedfull, 1);
    ptx::mbar_init(bar_seedfree, 1);
    ptx::fence_mbar_init();
  }
  if (warp == 2) { ptx::tmem_alloc2(ptx::smem_u32(s_tmem), 512); ptx::tmem_relinquish2(); }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync();
  ptx::tc_fence_after();
  const uint32_t tmem = *s_tmem;

  if (warp == 0) {
    // =========================== weight producer (both CTAs): this CTA's 8 KB half of every unit ===========
    uint32_t stage = 0, ph = 0;
    const int half_rows = (int)(p.pair_half_bytes >> 9);
    for (int st = 0; st < nst; ++st) {
      int row = (int)rank * half_rows;
      for (int j = 0; j < NS; ++j) {
        const int nu = bwd_step_units(j);
        for (int X = 0; X < 2; ++X) {
          int prow = row;
          for (int u = 0; u < nu; ++u) {
            ptx::mbar_wait(bar_wempty + 8 * stage, ph ^ 1);
            if (ptx::elect_one()) {
              if (leader) ptx::mbar_arrive_expect_tx(bar_wfull + 8 * stage, 2 * TC2_STAGE_BYTES);
              ptx::tma2_load_2d(sb + SM_WRING + stage * TC2_STAGE_BYTES, (const void*)&wmap, 0, prow, bar_wfull + 8 * stage);
            }
            __syncwarp();
            prow += (int)(TC2_STAGE_BYTES >> 9);
            if (++stage == TC2_NST) { stage = 0; ph ^= 1; }
          }
        }
        row += nu * (int)(TC2_STAGE_BYTES >> 9);
      }
    }
  } else if (warp == 1 && leader) {
    // =========================== MMA issuer (leader CTA) ===========================
    uint32_t stage = 0, ph = 0, actph0 = 0, actph1 = 0;
    const uint64_t adesc0 = ptx::umma_desc(sb, 1024, ptx::UMMA_SW128);
    const uint64_t bdesc0 = ptx::umma_desc(sb, 512, ptx::UMMA_SW64);
    const uint32_t tmem0 = __shfl_sync(0xffffffffu, tmem, 0);
    const uint32_t idesc = ptx::umma_idesc_f16(256, 256);
    for (int st = 0; st < nst; ++st) {
      for (int j = 0; j < NS; ++j) {
        const int nu = bwd_step_units(j);
        for (int X = 0; X < 2; ++X) {
          const uint32_t d_tmem = tmem0 + X * 256;
          // slot X's accumulator drained (and, for j >= 1, its A tile written) by both CTAs' epilogue warps
          if (X == 0) { ptx::mbar_wait_cluster(bar_act, actph0); actph0 ^= 1; }
          else { ptx::mbar_wait_cluster(bar_act + 8, actph1); actph1 ^= 1; }
          if (j == 0) ptx::mbar_wait_cluster(bar_seedfull, (uint32_t)X);        // one seed per (super-tile, slot): phase parity = X
          ptx::tc_fence_after();
          if (ptx::elect_one()) {
            uint32_t s_ = stage, ph_ = ph;
            const uint64_t bring = bdesc0 + (SM_WRING >> 4);
            uint32_t acc = 0u;
            if (j == 0) {
              const uint64_t aseed = adesc0 + (DG2_SEED >> 4);
#pragma unroll
              for (int kc = 0; kc < 4; ++kc) {
                while (!ptx::mbar_try_wait(bar_wfull + 8 * s_, ph_)) { }
                const uint64_t bd = bring + s_ * (TC2_STAGE_BYTES >> 4);
                const uint64_t ad = aseed + (uint64_t)((kc >> 1) * 1024 + (kc & 1) * 4);
                ptx::mma2_f16_ss(d_tmem, ad, bd, idesc, acc);
                ptx::mma2_f16_ss(d_tmem, ad + 2, bd + 2, idesc, 1u);
                acc = 1u;
                if (kc == 3) ptx::mma2_commit_mc(bar_seedfree, 3);
                ptx::mma2_commit_mc(bar_wempty + 8 * s_, 3);
                if (++s_ == TC2_NST) { s_ = 0; ph_ ^= 1; }
              }
            } else {
              const uint64_t aact = adesc0 + ((SM_ACT + X * 65536) >> 4);
#pragma unroll
              for (int kc = 0; kc < 8; ++kc) {
                while (!ptx::mbar_try_wait(bar_wfull + 8 * s_, ph_)) { }
                const uint64_t bd = bring + s_ * (TC2_STAGE_BYTES >> 4);
                const uint64_t ad = aact + (uint64_t)((kc >> 1) * 1024 + (kc & 1) * 4);
                ptx::mma2_f16_ss(d_tmem, ad, bd, idesc, acc);
                ptx::mma2_f16_ss(d_tmem, ad + 2, bd + 2, idesc, 1u);
                acc = 1u;
                ptx::mma2_commit_mc(bar_wempty + 8 * s_, 3);
                if (++s_ == TC2_NST) { s_ = 0; ph_ ^= 1; }
              }
            }
            ptx::mma2_commit_mc(bar_dfull + 8 * X, 3);
          }
          __syncwarp();
          stage += (uint32_t)nu;
          while (stage >= TC2_NST) { stage -= TC2_NST; ph ^= 1; }
        }
      }
    }
  } else if (warp == 3) {
    // =========================== seed loader (both CTAs): d_hv tile of (super-tile, slot) -> SEED ===========
    // the d_hv image (128 columns: in the record [half][K-block] pieces of 8 KB, in shared memory [K-block][half]) = four
    // 8 KB boxes of the gradient-record tensor map per (st, X); bytes of both CTAs are counted on the leader's barrier
    const int rec_rows = (int)(p.rec_grad >> 9);
    for (int st = 0; st < nst; ++st) {
      for (int X = 0; X < 2; ++X) {
        ptx::mbar_wait(bar_seedfree, (uint32_t)(X ^ 1));
        if (ptx::elect_one()) {
          if (leader) ptx::mbar_arrive_expect_tx(bar_seedfull, 2u * 32768u);
          const long long t = ((long long)vc * p.nst_plan + st) * 2 + X;
#pragma unroll
          for (int pc = 0; pc < 4; ++pc)                              // pc = half * 2 + kb  (record order)
            ptx::tma2_load_2d(sb + DG2_SEED + (uint32_t)(pc & 1) * 16384u + (uint32_t)(pc >> 1) * 8192u, (const void*)&gmap, 0, (int)(t * rec_rows) + pc * 16, bar_seedfull);
        }
        __syncwarp();
      }
    }
  } else if (warp >= 4) {
    // =========================== epilogue ===========================
    const int X = (warp - 4) >> 3, e = (warp - 4) & 7, q = warp & 3, ch = e >> 2;
    const int r = 32 * q + lane;
    const uint32_t t_lane = tmem + ((uint32_t)(32 * q) << 16) + X * 256;
    const uint32_t act_base = sb + SM_ACT + X * 65536;
    const float scale = loss_scale_from_absmax(__uint_as_float(*p.amax));
    arrive_leader(bar_act + 8 * X);                            // accumulator initially free
    uint32_t dph = 0;
    uint32_t swk[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) swk[c] = act_base + (uint32_t)(ch * 2) * 16384u + act_row_off(r) + (uint32_t)((c ^ (r & 7)) << 4);
    // gradient record: every warp copies ITS 32 rows of a K-block (4 KB, contiguous in the image) out as soon as it has written
    // them and, before it overwrites a K-block in the next step, waits for its own older copy to finish reading -- warp-local,
    // as in the forward's training mode (fused_tc2.cuh)
    const uint32_t slice = (uint32_t)q * 4096u;
    const uint64_t l2_first = ptx::l2_policy_evict_first();
    auto emit_gate = [&]() {
      if (lane == 0) ptx::bulk_wait_read1();
      __syncwarp();
    };
    auto emit_slice = [&](uint8_t* dst_img, int kb, uint32_t src_kblock) {
      ptx::fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        ptx::bulk_s2g_hint(dst_img + img_slice_off(q, kb, 256), src_kblock + slice, 4096u, l2_first);
        ptx::bulk_commit();
      }
    };
    const int nrows = plan_cta_rows(p.N, p.S, p.rays_per_cta, vc);
    const long long row_begin = (long long)vc * p.rays_per_cta * p.S;
    for (int st = 0; st < nst; ++st) {
      const int lr = st * TC_ST + X * TC_TILE + r;
      const bool valid = lr < nrows;
      const long long t = ((long long)vc * p.nst_plan + st) * 2 + X;
      const uint8_t* const mrec = p.mask + (size_t)t * p.rec_mask;
      uint8_t* const grec = p.grad + (size_t)t * p.rec_grad;
      const float dsig = valid ? p.d_raw[(row_begin + lr) * 4 + 3] * scale : 0.f;
      for (int j = 0; j < NS; ++j) {
        // ReLU mask of this step's output (the pre-activation of pts layer D - j), fetched before the wait
        uint4 mk = make_uint4(0u, 0u, 0u, 0u);
        if (j >= 1) mk = *reinterpret_cast<const uint4*>(mrec + (uint32_t)(D - j) * 4096u + (uint32_t)ch * 2048u + (uint32_t)r * 16u);
        ptx::mbar_wait(bar_dfull + 8 * X, dph);
        dph ^= 1;
        ptx::tc_fence_after();
        const int colw = ch * 128;
        uint32_t va[32], vb[32];
        ptx::tmem_ld_x32(t_lane + colw, va);
#pragma unroll
        for (int b = 0; b < 4; ++b) {
          const int col0 = colw + b * 32;
          uint32_t (&v)[32] = (b & 1) ? vb : va;
          uint32_t (&vn)[32] = (b & 1) ? va : vb;
          ptx::tmem_ld_wait();
          if (b < 3) ptx::tmem_ld_x32(t_lane + col0 + 32, vn);
          float x[32];
          as_float32(v, x);
          if (j == 1) {                                         // + d_sigma * alpha_linear.weight (run_nerf_helpers.py:106)
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float4 w = lds128(a_alpha + (uint32_t)(col0 + 4 * i) * 4u);
              x[4 * i + 0] = fmaf(dsig, w.x, x[4 * i + 0]); x[4 * i + 1] = fmaf(dsig, w.y, x[4 * i + 1]);
              x[4 * i + 2] = fmaf(dsig, w.z, x[4 * i + 2]); x[4 * i + 3] = fmaf(dsig, w.w, x[4 * i + 3]);
            }
          }
          if (j >= 1) {
            const uint32_t m = (b == 0) ? mk.x : (b == 1) ? mk.y : (b == 2) ? mk.z : mk.w;
#pragma unroll
            for (int i = 0; i < 32; ++i) x[i] = mask_apply(m, i, x[i]);
          }
          // next step's A operand, in place; batches 0, 1 fill K-block 2 ch, batches 2, 3 K-block 2 ch + 1
          if (b == 0) emit_gate();
          if (b == 2) {
            emit_slice(grec + rec_grad_step(j), 2 * ch, act_base + (uint32_t)(2 * ch) * 16384u);
            emit_gate();
          }
          if (b == 0) store_grad32_pre<0>(x, swk); else if (b == 1) store_grad32_pre<32>(x, swk);
          else if (b == 2) store_grad32_pre<64>(x, swk); else store_grad32_pre<96>(x, swk);
        }
        ptx::tc_fence_before();
        ptx::fence_proxy_async_smem();
        arrive_leader(bar_act + 8 * X);
        emit_slice(grec + rec_grad_step(j), 2 * ch + 1, act_base + (uint32_t)(2 * ch + 1) * 16384u);
      }
    }
    if (lane == 0) ptx::bulk_wait_all();
  }

  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync();
  if (warp == 2) ptx::tmem_dealloc2(tmem, 512);
}

// ---------------------------------------------------------------------------------------------------------------
// wgrad: layer-major.  Job = one weight block dW[Mc x Nc] = sum over tiles of A_t^T B_t, A = a gradient image (Mc
// columns, gradient record), B = an activation image (Nc columns, activation record); a contiguous range of CTAs
// serves a job, CTA g of G takes the job's tiles g, g + G, ...  Stage = one 64-row half tile of A and of B.
// 192 threads: warps 0-3 column sums (bias gradient) while streaming, then the TMEM epilogue; warp 4 producer; warp 5 issuer.
// ---------------------------------------------------------------------------------------------------------------
constexpr int WG2_THREADS = 192, WG2_MAX_STAGES = 4, WG2_MAX_JOBS = 16;
constexpr uint32_t WG2_BARS = 196608,                  // ring: 192 KB = 3 stages of a 256 + 256 column job
                   WG2_DSIG = WG2_BARS + 128, WG2_TOTAL = WG2_DSIG + 1024;

struct WgradJob {
  uint32_t a_off, b_off;        // image offsets inside the gradient / activation record
  int Mc, Nc;                   // columns of A (128 | 256) and of B (64 | 128 | 256)
  int cta0, ncta;               // CTA range serving this job
  float* db;                    // bias gradient (fp32, += scaled column sums of A) or NULL
  long long part_off;           // float offset of this job's partial blocks [ncta][Mc][Nc]
  int aux;                      // 1: A = d_hv  -> per-ray row sums into aux_dst [N,128] (view columns of views_linears[0])
                                // 2: B = h_{D-1} -> aux_dst[c] += sum_rows d_sigma[row] B[row][c]  (alpha_linear.weight), aux_b += sum d_sigma
  float* aux_dst; float* aux_b;
};
struct WgradParams {
  const uint8_t* act; const uint8_t* grad; uint32_t rec_act, rec_grad;
  long long N; int S, rays_per_cta, nst_plan; long long n_tiles;
  const unsigned int* amax; float* partial; const float* d_raw; int njobs;
  WgradJob jobs[WG2_MAX_JOBS];
};

__device__ __forceinline__ bool plan_tile_valid(const WgradParams& p, long long t) {
  const int cta = (int)(t / (2 * p.nst_plan)), st = (int)((t >> 1) % p.nst_plan);
  return st < plan_cta_nst(p.N, p.S, p.rays_per_cta, cta);
}

// (launched as 2-CTA clusters, so that its CTAs fill whole TPCs; launching it without clusters changes how its CTAs are
// placed on the SMs and would need its own measurement)
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(WG2_THREADS, 1) wgrad_tc_kernel(const WgradParams p) {
  uint8_t* smem = tc_smem;
  const uint32_t sb = ptx::smem_u32(smem);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if ((sb & 1023u) != 0) __trap();
  int ji = -1;
  for (int i = 0; i < p.njobs; ++i) if ((int)blockIdx.x >= p.jobs[i].cta0 && (int)blockIdx.x < p.jobs[i].cta0 + p.jobs[i].ncta) ji = i;
  if (ji < 0) return;                                   // (uniform per CTA, before any barrier / allocation)
  const WgradJob job = p.jobs[ji];
  const long long g = (int)blockIdx.x - job.cta0, G = job.ncta;        // 64-bit, as the tile indices they step
  const uint32_t bar_full = sb + WG2_BARS, bar_empty = sb + WG2_BARS + 32, bar_done = sb + WG2_BARS + 64;
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(smem + WG2_BARS + 96);
  if (threadIdx.x == 0) {
    for (int i = 0; i < WG2_MAX_STAGES; ++i) { ptx::mbar_init(bar_full + 8 * i, 1); ptx::mbar_init(bar_empty + 8 * i, 5); }
    ptx::mbar_init(bar_done, 1);
    ptx::fence_mbar_init();
  }
  if (warp == 0) { ptx::tmem_alloc(ptx::smem_u32(s_tmem), 512); ptx::tmem_relinquish(); }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem = *s_tmem;
  const int xkb = job.Mc >> 6, ykb = job.Nc >> 6;
  const uint32_t ybase = (uint32_t)xkb * 8192u;
  // ring: as many stages of this job's size as fit (narrow jobs get a 4th: the bytes in flight per SM set its share of the bus)
  const uint32_t stride = (uint32_t)(xkb + ykb) * 8192u;
  const uint32_t nstg = (WG2_BARS / stride < (uint32_t)WG2_MAX_STAGES) ? WG2_BARS / stride : (uint32_t)WG2_MAX_STAGES;
  long long my_halves = 0;
  for (long long t = g; t < p.n_tiles; t += G) if (plan_tile_valid(p, t)) my_halves += 2;

  if (warp == 4) {
    uint32_t s = 0, ph = 0;
    for (long long t = g; t < p.n_tiles; t += G) {
      if (!plan_tile_valid(p, t)) continue;
      for (int h = 0; h < 2; ++h) {
        ptx::mbar_wait(bar_empty + 8 * s, ph ^ 1);
        if (ptx::elect_one()) {
          ptx::mbar_arrive_expect_tx(bar_full + 8 * s, (uint32_t)(xkb + ykb) * 8192u);
          // 64-row half tile h of each operand: its K-blocks are adjacent in the record -> one contiguous piece per operand
          const uint8_t* xs = p.grad + (size_t)t * p.rec_grad + job.a_off + (size_t)h * xkb * 8192;
          const uint8_t* ys = p.act + (size_t)t * p.rec_act + job.b_off + (size_t)h * ykb * 8192;
          ptx::bulk_g2s(sb + s * stride, xs, (uint32_t)xkb * 8192u, bar_full + 8 * s);
          ptx::bulk_g2s(sb + s * stride + ybase, ys, (uint32_t)ykb * 8192u, bar_full + 8 * s);
        }
        __syncwarp();
        if (++s == nstg) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp == 5) {
    uint32_t s = 0, ph = 0;
    const uint32_t idesc = ptx::umma_idesc_f16_major(128, job.Nc, 1, 1);
    const int mhalves = job.Mc >> 7;
    for (long long i = 0; i < my_halves; ++i) {
      ptx::mbar_wait(bar_full + 8 * s, ph);
      ptx::tc_fence_after();
      if (ptx::elect_one()) {
        const uint32_t xb = sb + s * stride, yb = xb + ybase;
        for (int mh = 0; mh < mhalves; ++mh)
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            // MN-major SWIZZLE_128B (validated: nerf_b200_selftest_gemm_tn, tests of the tile-image wgrad): LBO = stride
            // between 64-column groups (8 KB: half-tile K-blocks), SBO = 1 KB (8-row groups), K step of 16 rows = 2 KB
            const uint64_t ad = ptx::umma_desc_full(xb + (uint32_t)(mh * 2) * 8192u + k * 2048, 8192, 1024, ptx::UMMA_SW128);
            const uint64_t bd = ptx::umma_desc_full(yb + k * 2048, 8192, 1024, ptx::UMMA_SW128);
            ptx::mma_f16_ss(tmem + mh * 256, ad, bd, idesc, (i > 0 || k > 0) ? 1u : 0u);
          }
        ptx::mma_commit(bar_empty + 8 * s);
        if (i == my_halves - 1) ptx::mma_commit(bar_done);
      }
      __syncwarp();
      if (++s == nstg) { s = 0; ph ^= 1; }
    }
  } else {
    // warps 0-3: while the tiles stream through shared memory -- bias gradient = column sums of the A half tiles; job
    // extras (aux): per-ray row sums of d_hv, or alpha_linear's weight gradient from the B tile; then the accumulator epilogue
    uint32_t s = 0, ph = 0;
    const int tid = threadIdx.x;                        // 0..127: columns 2 tid, 2 tid + 1
    const bool do_sum = (job.db != nullptr) && (2 * tid < job.Mc);
    const int c = 2 * tid;
    const uint32_t coff = (uint32_t)((c >> 6) * 8192 + (c & 7) * 2), cc = (uint32_t)((c & 63) >> 3);
    const float inv = 1.0f / loss_scale_from_absmax(__uint_as_float(*p.amax));
    float* s_dsig = reinterpret_cast<float*>(smem + WG2_DSIG);
    float s0 = 0.f, s1 = 0.f, a0 = 0.f, a1 = 0.f, bsum = 0.f;
    // aux == 2: d_sigma of a tile's 128 rows sits in shared memory (two slots); the NEXT tile's values are fetched while the
    // current tile is processed, so the global-load latency never sits between two stages
    auto load_dsig = [&](long long t_) -> float {
      const int cta_ = (int)(t_ / (2 * p.nst_plan)), st_ = (int)((t_ >> 1) % p.nst_plan), X_ = (int)(t_ & 1);
      const int lr_ = st_ * 256 + X_ * 128 + tid;
      return (lr_ < plan_cta_rows(p.N, p.S, p.rays_per_cta, cta_)) ? p.d_raw[((long long)cta_ * p.rays_per_cta * p.S + lr_) * 4 + 3] : 0.f;
    };
    auto next_valid = [&](long long t_) -> long long {
      for (t_ += G; t_ < p.n_tiles; t_ += G) if (plan_tile_valid(p, t_)) return t_;
      return -1;
    };
    int dslot = 0;
    if (job.aux == 2) {
      const long long t0 = next_valid(g - G);
      const float v = (t0 >= 0) ? load_dsig(t0) : 0.f;
      s_dsig[tid] = v;
      bsum += v;
      ptx::named_bar_sync(1, 128);
    }
    for (long long t = g; t < p.n_tiles; t += G) {
      if (!plan_tile_valid(p, t)) continue;
      const int cta = (int)(t / (2 * p.nst_plan)), st = (int)((t >> 1) % p.nst_plan), X = (int)(t & 1);
      const int nrows = plan_cta_rows(p.N, p.S, p.rays_per_cta, cta);
      const long long row_begin = (long long)cta * p.rays_per_cta * p.S;
      float v_next = 0.f;
      if (job.aux == 2) { const long long tn = next_valid(t); v_next = (tn >= 0) ? load_dsig(tn) : 0.f; }
      for (int h = 0; h < 2; ++h) {
        const int lr0 = st * 256 + X * 128 + h * 64;
        ptx::mbar_wait(bar_full + 8 * s, ph);
        // one row of this thread's column pair in a half-tile image that starts at shared-memory address `b_`
#define NB_LDPAIR(b_, r_, w_) asm volatile("ld.shared.b32 %0, [%1];" : "=r"(w_) : "r"((b_) + (uint32_t)(((r_) >> 3) * 1024 + ((r_) & 7) * 128) + ((cc ^ (uint32_t)((r_) & 7)) << 4)))
        // The stage is held only while its rows are copied into registers (64 LDS back to back); the arithmetic runs after the
        // release, while the producer already refills the stage (holding it through the sums cost 15 % of the kernel: measured)
        bool released = false;
        auto release = [&]() {
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(bar_empty + 8 * s);
          released = true;
        };
        if (do_sum || job.aux == 2) {
          const uint32_t abase = sb + s * stride + coff, bbase = abase + ybase;
          float h0 = 0.f, h1 = 0.f;                     // column sums of this half tile of A
          uint32_t wa[64];
#pragma unroll
          for (int r = 0; r < 64; ++r) NB_LDPAIR(abase, r, wa[r]);
          if (job.aux == 2) {
            // A = d_feat (bias gradient) and B = h_{D-1} (x d_sigma -> alpha_linear.weight)
            uint32_t wb[64];
#pragma unroll
            for (int r = 0; r < 64; ++r) NB_LDPAIR(bbase, r, wb[r]);
            release();
            const float* ds = s_dsig + dslot * 128 + h * 64;
            float a0b = 0.f, a1b = 0.f;
#pragma unroll
            for (int r = 0; r < 64; r += 2) {
              const __half2 hb0 = *reinterpret_cast<const __half2*>(&wb[r]), hb1 = *reinterpret_cast<const __half2*>(&wb[r + 1]);
              const float d0 = ds[r], d1 = ds[r + 1];
              a0 = fmaf(d0, __low2float(hb0), a0); a1 = fmaf(d0, __high2float(hb0), a1);
              a0b = fmaf(d1, __low2float(hb1), a0b); a1b = fmaf(d1, __high2float(hb1), a1b);
            }
            a0 += a0b; a1 += a1b;
          } else if (!(job.aux == 1 && p.S % 64 != 0)) {
            release();                                  // (aux == 1 with S % 64 != 0 may have to walk the rows again: keeps the stage)
          }
          {
            float e0 = 0.f, e1 = 0.f, o0 = 0.f, o1 = 0.f;
#pragma unroll
            for (int r = 0; r < 64; r += 2) {
              const __half2 ha = *reinterpret_cast<const __half2*>(&wa[r]), hb = *reinterpret_cast<const __half2*>(&wa[r + 1]);
              e0 += __low2float(ha); e1 += __high2float(ha);
              o0 += __low2float(hb); o1 += __high2float(hb);
            }
            h0 = e0 + o0; h1 = e1 + o1;
          }
          s0 += h0; s1 += h1;
          if (job.aux == 1 && do_sum) {
            // per-ray row sums of d_hv.  Rows past the CTA's range are zero in the image (dhv_seed_kernel), so when the valid
            // rows of this half tile belong to ONE ray (always for S % 64 == 0) its sum is the half-tile column sum
            const int nvalid = (nrows - lr0 < 64) ? nrows - lr0 : 64;
            if (nvalid > 0) {
              const long long m0 = row_begin + lr0;                     // row_begin is a multiple of S: rays are whole per CTA
              const long long ray_a = (long long)cta * p.rays_per_cta + lr0 / p.S, ray_b = (long long)cta * p.rays_per_cta + (lr0 + nvalid - 1) / p.S;
              if (ray_a == ray_b) {
                atomicAdd(job.aux_dst + ray_a * 128 + c, h0 * inv); atomicAdd(job.aux_dst + ray_a * 128 + c + 1, h1 * inv);
              } else {                                  // general S: walk the rows, flush at every ray boundary
                long long ray = ray_a;
                int left = (int)((ray + 1) * p.S - m0);
                float r0 = 0.f, r1 = 0.f;
                for (int r = 0; r < nvalid; ++r) {
                  uint32_t w;
                  NB_LDPAIR(abase, r, w);
                  const __half2 hh = *reinterpret_cast<const __half2*>(&w);
                  r0 += __low2float(hh); r1 += __high2float(hh);
                  if (--left == 0 || r == nvalid - 1) {
                    atomicAdd(job.aux_dst + ray * 128 + c, r0 * inv); atomicAdd(job.aux_dst + ray * 128 + c + 1, r1 * inv);
                    r0 = r1 = 0.f; ++ray; left = p.S;
                  }
                }
              }
            }
          }
        }
#undef NB_LDPAIR
        if (!released) release();
        if (++s == nstg) { s = 0; ph ^= 1; }
      }
      if (job.aux == 2) {                               // the prefetched d_sigma of the next tile -> the other slot
        s_dsig[(dslot ^ 1) * 128 + tid] = v_next;
        bsum += v_next;
        dslot ^= 1;
        ptx::named_bar_sync(1, 128);
      }
    }
    if (job.aux == 2 && my_halves > 0) {
      atomicAdd(job.aux_dst + c, a0); atomicAdd(job.aux_dst + c + 1, a1);
      bsum = warp_sum(bsum);
      if (lane == 0) atomicAdd(job.aux_b, bsum);
    }
    if (do_sum && my_halves > 0) { atomicAdd(job.db + c, s0 * inv); atomicAdd(job.db + c + 1, s1 * inv); }
    float* part = p.partial + job.part_off + (size_t)g * job.Mc * job.Nc;
    if (my_halves > 0) {
      ptx::mbar_wait(bar_done, 0);
      ptx::tc_fence_after();
    }
    const int r = 32 * warp + lane;
    for (int mh = 0; mh < (job.Mc >> 7); ++mh)
      for (int c0 = 0; c0 < job.Nc; c0 += 32) {
        uint32_t v[32];
        if (my_halves > 0) {
          ptx::tmem_ld_x32(tmem + ((uint32_t)(32 * warp) << 16) + mh * 256 + c0, v);
          ptx::tmem_ld_wait();
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = 0u;
        }
        float4* o = reinterpret_cast<float4*>(part + (size_t)(mh * 128 + r) * job.Nc + c0);
#pragma unroll
        for (int j = 0; j < 8; ++j)
          o[j] = make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]), __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
      }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 0) ptx::tmem_dealloc(tmem, 512);
}

// dst[o][i] += inv_scale * sum_g partial[g][o][i]   (i < n_valid; dst row stride ldw)
struct ReduceJob { long long part_off; int ncta, Mc, Nc, n_valid, ldw; float* dst; };
struct ReduceParams { const float* partial; const unsigned int* amax; int njobs; ReduceJob jobs[WG2_MAX_JOBS]; };

__global__ void __launch_bounds__(256) wgrad_reduce_kernel(const ReduceParams p) {
  const ReduceJob j = p.jobs[blockIdx.y];
  const int idx = blockIdx.x * 256 + threadIdx.x;
  if (idx >= j.Mc * j.Nc) return;
  const int o = idx / j.Nc, i = idx - o * j.Nc;
  if (i >= j.n_valid) return;
  const float* src = p.partial + j.part_off + idx;
  float s = 0.f;
  for (int g = 0; g < j.ncta; ++g) s += src[(size_t)g * j.Mc * j.Nc];
  const float inv = 1.0f / loss_scale_from_absmax(__uint_as_float(*p.amax));
  j.dst[(size_t)o * j.ldw + i] += s * inv;
}

// ---------------------------------------------------------------------------------------------------------------
// the view columns of views_linears[0] (alpha_linear and the per-ray sums of d_hv ride along in the wgrad kernel, whose tiles
// already hold their operands; rgb_linear's gradient comes from dhv_seed_heads_kernel)
// ---------------------------------------------------------------------------------------------------------------
// views_linears[0].weight[c][W + e] += sum_rays dsum[ray][c] * gamma(viewdir_ray)[e]      (run_nerf_helpers.py:108-110);
// block e == ICV: dbv[c] += sum_rays dsum[ray][c]  (this pass's bias gradient of views_linears[0], for the kernel below)
__global__ void __launch_bounds__(128) views_enc_wgrad_kernel(const float* __restrict__ dsum, const float* __restrict__ encv, long long N, int ICV,
                                                            float* __restrict__ views_w, int ld, int col0, float* __restrict__ dbv) {
  const int e = blockIdx.x, c = threadIdx.x;
  const long long n0 = (long long)blockIdx.y * 64, n1 = (n0 + 64 < N) ? n0 + 64 : N;
  float s = 0.f;
  if (e < ICV) {
    for (long long n = n0; n < n1; ++n) s = fmaf(dsum[n * 128 + c], encv[n * ICV + e], s);
    atomicAdd(views_w + (size_t)c * ld + col0 + e, s);
  } else {
    for (long long n = n0; n < n1; ++n) s += dsum[n * 128 + c];
    atomicAdd(dbv + c, s);
  }
}

// views_linears[0].weight[v][f] (f < W) += sum_k G[v][k] W_feat[f][k] + dbv[v] b_feat[f], with G = d_hv^T h_{D-1} (the views job of
// the wgrad kernel, already reduced and un-scaled): the feature layer has no activation, so
//   d_hv^T feat = d_hv^T (h_{D-1} W_feat^T + 1 b_feat^T) = G W_feat^T + (sum_rows d_hv) b_feat^T
// and feature_linear's output never has to be stored (run_nerf_helpers.py:107-110).  grid = 128 (v), block = 256 (f).
__global__ void __launch_bounds__(256) views_feat_wgrad_kernel(const float* __restrict__ G, const float* __restrict__ dbv, const float* __restrict__ feat_w,
                                                             const float* __restrict__ feat_b, float* __restrict__ views_w, int ld) {
  __shared__ float s_g[256];
  const int v = blockIdx.x, f = threadIdx.x;
  s_g[f] = G[v * 256 + f];
  __syncthreads();
  const float4* w4 = reinterpret_cast<const float4*>(feat_w + (size_t)f * 256);
  float acc = dbv[v] * feat_b[f];
#pragma unroll 8
  for (int k4 = 0; k4 < 64; ++k4) {
    const float4 w = w4[k4];
    acc = fmaf(s_g[4 * k4], w.x, acc); acc = fmaf(s_g[4 * k4 + 1], w.y, acc); acc = fmaf(s_g[4 * k4 + 2], w.z, acc); acc = fmaf(s_g[4 * k4 + 3], w.w, acc);
  }
  views_w[(size_t)v * ld + f] += acc;
}

}  // namespace nb
