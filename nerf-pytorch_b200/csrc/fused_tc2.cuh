// fused_tc2.cuh -- CTA-pair (cta_group::2) version of the fused network pass.
//
// Two CTAs of a cluster (a TPC's SM pair) work as one: every tcgen05.mma covers M = 256 rows -- 128 rows of
// each CTA's own A tile, accumulated in each CTA's own TMEM -- while the B operand (the weight chunk) is split
// across the pair, so a K=32 chunk costs 8 KB of shared memory and 8 KB of L2->SM traffic per SM instead of 16.
// The freed ring space (6 stages x 8 KB) pays for a tile-major schedule: per layer the leader CTA issues ALL
// chunks of slot A's pair-tile (17 MMAs back to back), then all chunks of slot B's; slot A's epilogue (TMEM
// drain, ReLU, fp16, next layer's A tile) runs on both CTAs while the tensor pipes work on slot B, and vice
// versa -- the lock-step kernel (fused_tc.cuh) leaves the tensor pipe idle during both epilogues.
// Everything else (sampler, epilogue math, heads, compositing) is the code of fused_tc.cuh, per CTA.
//
// Cross-CTA protocol (barriers live at the same shared-memory offset in both CTAs):
//   w_full[7]  leader  : both CTAs' tensor-map TMA loads (cta_group::2) count their bytes here (expect_tx = 2 x 8 KB)
//   w_empty[7] both    : tcgen05.commit.cta_group::2 multicast -> both producers may refill the stage
//   d_full[2]  both    : multicast commit -> both CTAs' epilogue warps of that slot
//   act[2]     leader  : 16 arrivals = one per epilogue warp of the slot, 8 local + 8 remote (accumulator drained, A tile written)
//   enc_full   leader  : 2 arrivals (both sampler warps);  enc_free both: multicast commit after the last encoding chunk
// Training mode (template parameter EMIT, train_common.cuh): every post-ReLU A tile the epilogue writes (h_l) is also copied to
// the tile's record in global memory with cp.async.bulk shared -> global, one 16 KB K-block at a time, each as soon as the four
// warps that own it have written it; the next layer's epilogue waits per K-block (cp.async.bulk.wait_group.read) before it
// overwrites the tile in place.  The view layer's output goes out straight from the registers as 32-byte sectors
// (store_img32_global; for the 64 KB tiles that costs more LSU time than it saves: measured).  The sign bits of the
// pre-activations go out as one 16-byte store per thread and layer; the encodings are bulk-copied by the sampler warp.
#pragma once
#include <cuda.h>
#include "fused_tc.cuh"
#include "train_common.cuh"

namespace nb {

constexpr int TC2_NST = 7;                       // ring stages; one stage (unit) = 8 KB = one TMA box, one barrier pair
constexpr uint32_t TC2_STAGE_BYTES = 8192;
// shared-memory map behind the ring (ACT / ENC / WRING start as in fused_tc.cuh): the pair kernel needs only its
// N-half of the resident bias operand and parks the head partials in the (dead) A tile, which pays for the
// 7th stage.  With 7 x 8 KB in flight and a release -> refill -> ready round trip of ~1.4 k cycles the stream
// sustains one unit per ~240 cycles (consumption: 257); 3 x 16 KB sustained one per ~325.
constexpr uint32_t P2_ONES = SM_WRING + TC2_NST * TC2_STAGE_BYTES;   // 221184: 2 x 256 B bias-selector atoms
constexpr uint32_t P2_BIASB = P2_ONES + 512;                          // 221696: 4 KB, this CTA's rows of the bias operand
constexpr uint32_t P2_HEADS = P2_BIASB + TC_BIAS_CHUNK_BYTES / 2;     // 225792: head weights
constexpr uint32_t P2_BARS = P2_HEADS + 4128;                         // 229920: mbarriers
constexpr uint32_t P2_MISC = P2_BARS + 256;                           // 230176: tmem ptr, compositing carry, pass counter
constexpr uint32_t P2_TOTAL = P2_MISC + 128;                          // 230304

// training-mode save buffers of one pass (train_common.cuh)
struct TrainSaveDev { uint8_t* act; uint8_t* mask; int nst_plan; uint32_t rec_act, rec_mask; };
static_assert(P2_TOTAL <= SM_ALLOC, "pair kernel shared-memory map exceeds the allocation");

// ring units per pass of layer l (all even)
__host__ __device__ __forceinline__ int tc2_layer_units(int l, int D, int skip) {
  const int nch = tc_layer_chunks(l, D, skip);
  return (l == D + 1) ? nch / 2 : nch;
}

template <bool EMIT>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(TC_THREADS, 1) march_tc2_kernel(const MarchParams p, const __grid_constant__ CUtensorMap wmap,
                                                                                          const TrainSaveDev sv) {
  uint8_t* smem = tc_smem;
  const uint32_t sb = ptx::smem_u32(smem);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if ((sb & 1023u) != 0) __trap();
  const uint32_t rank = ptx::cluster_ctarank();
  const bool leader = (rank == 0);

  float* s_heads = reinterpret_cast<float*>(smem + P2_HEADS);
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(smem + P2_MISC);
  const uint32_t a_heads = sb + P2_HEADS, a_carry = sb + P2_MISC + 16, a_pass = sb + P2_MISC + 64;

  // mbarriers (same offsets in both CTAs)
  const uint32_t bar_wfull = sb + P2_BARS;            // [7] (leader)
  const uint32_t bar_wempty = sb + P2_BARS + 56;      // [7]
  const uint32_t bar_dfull = sb + P2_BARS + 112;      // [2]
  const uint32_t bar_act = sb + P2_BARS + 128;        // [2] (leader)
  const uint32_t bar_encfull = sb + P2_BARS + 144;    //     (leader)
  const uint32_t bar_encfree = sb + P2_BARS + 152;
  // arrive on a barrier that lives in the leader CTA
  // One arrival per warp; every lane has fenced its own writes (fence.proxy.async) before the __syncwarp.  The peer's
  // data is consumed by the peer SM's own tensor core, so the remote arrive needs no cluster-scope release.
  auto arrive_leader = [&](uint32_t bar) {
    __syncwarp();
    if (lane == 0) {
      if (leader) ptx::mbar_arrive(bar);
      else ptx::mbar_arrive_remote(ptx::mapa(bar, 0));
    }
  };

  // this CTA's rays / rows; both CTAs of a pair run the same number of super-tiles
  const long long ray0 = (long long)blockIdx.x * p.rays_per_cta;
  const long long ray1 = (ray0 + p.rays_per_cta < p.N) ? ray0 + p.rays_per_cta : p.N;
  const int nrows = (ray1 > ray0) ? (int)(ray1 - ray0) * p.S : 0;
  const long long pray0 = (long long)(blockIdx.x ^ 1) * p.rays_per_cta;
  const long long pray1 = (pray0 + p.rays_per_cta < p.N) ? pray0 + p.rays_per_cta : p.N;
  const int prows = (pray1 > pray0) ? (int)(pray1 - pray0) * p.S : 0;
  const int nst = ((nrows > prows ? nrows : prows) + TC_ST - 1) / TC_ST;
  const long long row_begin = ray0 * p.S;
  const int D = p.D, NL = p.D + (p.use_viewdirs ? 2 : 0);
  const int last_enc_layer = (p.skip >= 0 && p.skip + 1 < D) ? p.skip + 1 : 0;

  // ---- one-time setup ----
  const int n_bias = D + (p.use_viewdirs ? 1 : 0);
  if (threadIdx.x < 16) write_bias_selector(sb + P2_ONES + (threadIdx.x >> 3) * 256, threadIdx.x & 7, 0, n_bias);
  // this CTA's half (rows 128*rank ..) of the resident bias operand
  for (int i = threadIdx.x; i < (int)(TC_BIAS_CHUNK_BYTES / 32); i += TC_THREADS)
    reinterpret_cast<uint4*>(smem + P2_BIASB)[i] = reinterpret_cast<const uint4*>(p.biasb + rank * (TC_BIAS_CHUNK_BYTES / 2))[i];
  ptx::fence_proxy_async_smem();
  for (int i = threadIdx.x; i < HEADS_FLOATS; i += TC_THREADS) s_heads[i] = p.heads[i];
  if (threadIdx.x == 0) {
    sts32(a_carry + CARRY_T, 1.0f); sts32(a_carry + CARRY_R, 0.f); sts32(a_carry + CARRY_G, 0.f); sts32(a_carry + CARRY_B, 0.f);
    sts32(a_carry + CARRY_D, 0.f); sts32(a_carry + CARRY_A, 0.f); st_release_shared(a_carry + CARRY_TURN, 0u); st_release_shared(a_pass, 0u);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < TC2_NST; ++i) { ptx::mbar_init(bar_wfull + 8 * i, 1); ptx::mbar_init(bar_wempty + 8 * i, 1); }
    for (int x = 0; x < 2; ++x) { ptx::mbar_init(bar_dfull + 8 * x, 1); ptx::mbar_init(bar_act + 8 * x, 16); }
    ptx::mbar_init(bar_encfull, 2);
    ptx::mbar_init(bar_encfree, 2);
    ptx::fence_mbar_init();
  }
  if (warp == 2) { ptx::tmem_alloc2(ptx::smem_u32(s_tmem), 512); ptx::tmem_relinquish2(); }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync();                                  // peer barriers initialised before any remote arrive
  ptx::tc_fence_after();
  const uint32_t tmem = *s_tmem;

  if (warp == 0) {
    // =========================== weight producer (both CTAs): this CTA's half of every unit ===========
    // unit = one 8 KB ring stage = one TMA box of 16 stream rows: one chunk half of an N=256 layer, or two
    // consecutive chunk halves (2 x 4 KB) of the N=128 view layer
    uint32_t stage = 0, ph = 0;
    const int half_rows = (int)(p.pair_half_bytes >> 9);     // rows (512 B) of one rank's stream
    for (int st = 0; st < nst; ++st) {
      int row = (int)rank * half_rows;
      for (int l = 0; l < NL; ++l) {
        const int nu = tc2_layer_units(l, D, p.skip);
        for (int X = 0; X < 2; ++X) {                               // pass of slot A, then the same units again for slot B
          int prow = row;
          for (int u = 0; u < nu; ++u) {
            ptx::mbar_wait(bar_wempty + 8 * stage, ph ^ 1);
            if (ptx::elect_one()) {
              // every load (cta_group::2) counts its bytes on the LEADER's w_full, which expects both CTAs' boxes
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
    // =========================== MMA issuer (leader CTA, one warp) ===========================
    // A whole pass (all units of one slot's layer: 17-21 MMAs) is issued by ONE elected lane inside ONE elected
    // region; the w_full waits and the w_empty / d_full commits of the pass happen inside it.  Measured
    // (tools/issue_probe2.py): every entry into an elect_one() region costs the tensor pipe ~85 idle cycles,
    // whatever else the iteration does -- bursts of 2 / 4 / 8 MMAs per region run at 76 % / 86 % / 97 % of the
    // back-to-back rate, commits are free and a (ready) mbarrier wait costs ~33 cycles.  Earlier versions of
    // this kernel entered a region per ring stage (4 MMAs) and were issue-bound at ~645 cycles per 515 of MMA.
    uint32_t stage = 0, ph = 0, actph0 = 0, actph1 = 0;
    const uint64_t adesc0 = ptx::umma_desc(sb, 1024, ptx::UMMA_SW128);
    const uint64_t bdesc0 = ptx::umma_desc(sb, 512, ptx::UMMA_SW64);
    const uint64_t bias_desc = ptx::umma_desc(sb + P2_BIASB, 256, ptx::UMMA_SW32);
    const uint32_t tmem0 = __shfl_sync(0xffffffffu, tmem, 0);
    for (int st = 0; st < nst; ++st) {
      ptx::mbar_wait_cluster(bar_encfull, st & 1);
      for (int l = 0; l < NL; ++l) {
        const int nu = tc2_layer_units(l, D, p.skip);
        const bool view_layer = (l == D + 1);
        const bool skip_layer = (l < D && p.skip >= 0 && l == p.skip + 1);
        const bool has_bias = tc_layer_has_bias(l, D);
        const uint32_t idesc = ptx::umma_idesc_f16(256, view_layer ? 128 : 256);
        for (int X = 0; X < 2; ++X) {
          const uint32_t d_tmem = tmem0 + X * 256;
          const uint64_t sel_desc = ptx::umma_desc(sb + P2_ONES + X * 256, 0, ptx::UMMA_SW32);
          // slot X's accumulator drained and its A tile written by both CTAs' epilogue warps
          if (X == 0) { ptx::mbar_wait_cluster(bar_act, actph0); actph0 ^= 1; }
          else { ptx::mbar_wait_cluster(bar_act + 8, actph1); actph1 ^= 1; }
          ptx::tc_fence_after();
          if (ptx::elect_one()) {
            // Everything between two MMAs of the issuing thread is exposed tensor-pipe idle time (the queue is
            // shallow), so the per-unit work is kept to: one try_wait, one multiply-add for the stage's B
            // descriptor, the MMAs, one commit.  A-descriptor offsets are compile-time (unrolled loops).
            uint32_t s_ = stage, ph_ = ph;
            const uint64_t bring = bdesc0 + (SM_WRING >> 4);
            uint32_t acc = has_bias ? 1u : 0u;
            if (has_bias) ptx::mma2_f16_ss(d_tmem, sel_desc, bias_desc, idesc, 0u);
            if (l == 0 || skip_layer) {
              const uint64_t aenc = adesc0 + ((SM_ENC + X * 16384) >> 4);
#pragma unroll
              for (int c = 0; c < 2; ++c) {
                while (!ptx::mbar_try_wait(bar_wfull + 8 * s_, ph_)) { }
                const uint64_t bd = bring + s_ * (TC2_STAGE_BYTES >> 4);
                ptx::mma2_f16_ss(d_tmem, aenc + c * 4, bd, idesc, acc);
                ptx::mma2_f16_ss(d_tmem, aenc + c * 4 + 2, bd + 2, idesc, 1u);
                acc = 1u;
                if (c == 1 && l == last_enc_layer) ptx::mma2_commit_mc(bar_encfree, 3);
                ptx::mma2_commit_mc(bar_wempty + 8 * s_, 3);
                if (++s_ == TC2_NST) { s_ = 0; ph_ ^= 1; }
              }
            }
            const uint64_t aact = adesc0 + ((SM_ACT + X * 65536) >> 4);
            if (l != 0 && !view_layer) {
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
            } else if (view_layer) {
#pragma unroll
              for (int u = 0; u < 4; ++u) {
                while (!ptx::mbar_try_wait(bar_wfull + 8 * s_, ph_)) { }
                const uint64_t bd = bring + s_ * (TC2_STAGE_BYTES >> 4);
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                  const int kc = 2 * u + h;
                  const uint64_t ad = aact + (uint64_t)((kc >> 1) * 1024 + (kc & 1) * 4);
                  ptx::mma2_f16_ss(d_tmem, ad, bd + h * 256, idesc, acc);
                  ptx::mma2_f16_ss(d_tmem, ad + 2, bd + h * 256 + 2, idesc, 1u);
                  acc = 1u;
                }
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
  } else if (warp == 2 && leader) {
    // idle (the second issuer warp of the single-CTA kernel)
  } else if ((warp == 1 || warp == 2) && !leader) {
    // idle: the peer's bulk copies signal the leader's w_full barriers directly
  } else if (warp >= 4) {
    // =========================== epilogue ===========================
    // TMEM lane quadrant is fixed by (warp id % 4)
    const int X = (warp - 4) >> 3, e = (warp - 4) & 7, q = warp & 3, ch = e >> 2;
    const int r = 32 * q + lane;                                  // tile row == TMEM lane
    const uint32_t t_lane = tmem + ((uint32_t)(32 * q) << 16) + X * 256;
    const uint32_t act_base = sb + SM_ACT + X * 65536;
    arrive_leader(bar_act + 8 * X);                            // accumulator initially free
    uint32_t dph = 0;
    // swizzled 16-byte-chunk addresses of this thread's row in the two K-blocks of its column half
    uint32_t swk[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) swk[c] = act_base + (uint32_t)(ch * 2) * 16384u + act_row_off(r) + (uint32_t)((c ^ (r & 7)) << 4);
    // Compositing of super-tile s is deferred to the idle window after this slot's layer-1 epilogue of super-tile
    // s + 1 (the epilogue warps wait ~3.5 k cycles for every d_full): done right after the heads it delayed the
    // next super-tile's layer-0 epilogue and left the tensor pipes idle for ~7 k cycles per super-tile.
    // The raw values wait in registers (ch == 0 warps), row indices are recomputed.
    float4 pend = make_float4(0.f, 0.f, 0.f, 0.f);
    auto composite_st = [&](int s) {
      const int lr_ = s * TC_ST + X * TC_TILE + r;
      const bool valid_ = lr_ < nrows;
      const int rl_ = (valid_ ? lr_ : nrows - 1) / p.S;
      long long nr_ = ray0 + rl_;
      if (nr_ > p.N - 1) nr_ = p.N - 1;
      if (nr_ < 0) nr_ = 0;
      composite_rows(p, pend, valid_, lr_, rl_, nr_, row_begin, s, X, q, lane, a_carry);
    };
    const int defer_l = (NL > 1) ? 1 : 0;
    // training mode: every warp copies ITS 32 rows of a K-block (4 KB, contiguous in the image) to the record as soon as it has
    // written them -- cp.async.bulk shared -> global issued by lane 0, one bulk group per slice -- and before it overwrites a
    // K-block in the next layer it waits for its own older copy to finish reading (wait_group.read 1: the newer group, the
    // other K-block, may still be pending).  Nothing here crosses a warp: no barrier joins the epilogue warps.
    const uint32_t slice = (uint32_t)q * 4096u;
    const uint64_t l2_first = EMIT ? ptx::l2_policy_evict_first() : 0ull;      // records are written once, read once by the backward
    auto emit_gate = [&](bool all) {
      if (lane == 0) { if (all) ptx::bulk_wait_read0(); else ptx::bulk_wait_read1(); }
      __syncwarp();
    };
    // dst_img: the image in the record, kb: its K-block, C: its columns; src_kblock: the K-block in shared memory
    auto emit_slice = [&](uint8_t* dst_img, int kb, int C, uint32_t src_kblock) {
      ptx::fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        ptx::bulk_s2g_hint(dst_img + img_slice_off(q, kb, C), src_kblock + slice, 4096u, l2_first);
        ptx::bulk_commit();
      }
    };
    for (int st = 0; st < nst; ++st) {
      float hp0 = 0.f, hp1 = 0.f, hp2 = 0.f, hp3 = 0.f;           // head partial sums of this thread's columns
      uint8_t* const arec = EMIT ? sv.act + (size_t)((blockIdx.x * sv.nst_plan + st) * 2 + X) * sv.rec_act : nullptr;
      uint8_t* const mrec = EMIT ? sv.mask + (size_t)((blockIdx.x * sv.nst_plan + st) * 2 + X) * sv.rec_mask : nullptr;
      const int lr = st * TC_ST + X * TC_TILE + r;                // row index inside this CTA's range
      const bool valid = lr < nrows;
      const int rl = (valid ? lr : nrows - 1) / p.S;              // local ray
      long long n_ray = ray0 + rl;
      if (n_ray > p.N - 1) n_ray = p.N - 1;                       // (padding CTA of an odd pair / empty range)
      if (n_ray < 0) n_ray = 0;
      for (int l = 0; l < NL; ++l) {
        ptx::mbar_wait(bar_dfull + 8 * X, dph);
        dph ^= 1;
        ptx::tc_fence_after();
        if (l <= D) {
          // pts layer (ReLU) or feature layer (no activation): 128 columns per warp in 4 batches,
          // the TMEM load of batch b+1 in flight while batch b is converted and stored
          const bool last_pts = (l == D - 1);
          const bool write_act = !(last_pts && !p.use_viewdirs);
          const int colw = ch * 128;
          uint32_t va[32], vb[32];
          uint32_t mk[4] = {0u, 0u, 0u, 0u};                       // EMIT: sign bits of this thread's 128 pre-activations
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
            if (EMIT && l < D) {
#pragma unroll
              for (int j = 0; j < 32; ++j) mk[b] = mask_push(mk[b], x[j]);
            }
            if (last_pts) {
              if (p.use_viewdirs) {                               // alpha_linear (run_nerf_helpers.py:106)
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                  const float4 w = lds128(a_heads + (uint32_t)(col0 + 4 * j) * 4u);
                  hp3 = fmaf(fmaxf(x[4 * j + 0], 0.f), w.x, hp3); hp3 = fmaf(fmaxf(x[4 * j + 1], 0.f), w.y, hp3);
                  hp3 = fmaf(fmaxf(x[4 * j + 2], 0.f), w.z, hp3); hp3 = fmaf(fmaxf(x[4 * j + 3], 0.f), w.w, hp3);
                }
              } else {                                            // output_linear (:117)
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                  const float4 w0 = lds128(a_heads + (uint32_t)(col0 + 4 * j) * 4u), w1 = lds128(a_heads + (uint32_t)(256 + col0 + 4 * j) * 4u);
                  const float4 w2 = lds128(a_heads + (uint32_t)(512 + col0 + 4 * j) * 4u), w3 = lds128(a_heads + (uint32_t)(768 + col0 + 4 * j) * 4u);
                  const float h0 = fmaxf(x[4 * j + 0], 0.f), h1 = fmaxf(x[4 * j + 1], 0.f), h2 = fmaxf(x[4 * j + 2], 0.f), h3 = fmaxf(x[4 * j + 3], 0.f);
                  hp0 = fmaf(h0, w0.x, hp0); hp0 = fmaf(h1, w0.y, hp0); hp0 = fmaf(h2, w0.z, hp0); hp0 = fmaf(h3, w0.w, hp0);
                  hp1 = fmaf(h0, w1.x, hp1); hp1 = fmaf(h1, w1.y, hp1); hp1 = fmaf(h2, w1.z, hp1); hp1 = fmaf(h3, w1.w, hp1);
                  hp2 = fmaf(h0, w2.x, hp2); hp2 = fmaf(h1, w2.y, hp2); hp2 = fmaf(h2, w2.z, hp2); hp2 = fmaf(h3, w2.w, hp2);
                  hp3 = fmaf(h0, w3.x, hp3); hp3 = fmaf(h1, w3.y, hp3); hp3 = fmaf(h2, w3.z, hp3); hp3 = fmaf(h3, w3.w, hp3);
                }
              }
            }
            if (write_act) {
              if (EMIT) {
                // batches 0, 1 fill K-block 2 ch, batches 2, 3 K-block 2 ch + 1 (the previous layer's copies: one group each, in this order)
                if (b == 0) emit_gate(false);
                if (b == 2) {
                  if (l < D) emit_slice(arec + rec_act_h(l), 2 * ch, 256, act_base + (uint32_t)(2 * ch) * 16384u);
                  emit_gate(l == D);                            // (l == D: nothing was committed in between -> drain everything)
                }
              }
              // (b & 1) selects the K-block inside the column half; ch selects the half: the
              // immediate part of the address is compile-time, the row/swizzle part is in sw[]
              if (l < D) {
                if (b == 0) store_act32_pre<true, 0>(x, swk); else if (b == 1) store_act32_pre<true, 32>(x, swk);
                else if (b == 2) store_act32_pre<true, 64>(x, swk); else store_act32_pre<true, 96>(x, swk);
              } else {
                if (b == 0) store_act32_pre<false, 0>(x, swk); else if (b == 1) store_act32_pre<false, 32>(x, swk);
                else if (b == 2) store_act32_pre<false, 64>(x, swk); else store_act32_pre<false, 96>(x, swk);
              }
            }
          }
          // this slot's bias selector for the NEXT layer
          {
            const int nxt = (l + 1 < n_bias) ? l + 1 : ((l == NL - 1) ? 0 : -1);
            if (q == 0 && ch == 0 && lane < 8 && nxt >= 0) write_bias_selector(sb + P2_ONES + X * 256, lane, nxt, n_bias);
          }
          ptx::tc_fence_before();
          ptx::fence_proxy_async_smem();
          arrive_leader(bar_act + 8 * X);
          if (EMIT) {
            if (l < D) *reinterpret_cast<uint4*>(mrec + (uint32_t)l * 4096u + (uint32_t)ch * 2048u + (uint32_t)r * 16u) = make_uint4(mk[0], mk[1], mk[2], mk[3]);
            // second K-block of h_l (feature_linear's output, l == D, is not recorded)
            if (l < D && write_act) emit_slice(arec + rec_act_h(l), 2 * ch + 1, 256, act_base + (uint32_t)(2 * ch + 1) * 16384u);
          }
        } else {
          // views_linears[0] (N=128): 64 columns per warp; + per-ray view bias, ReLU, rgb_linear
          const float* vbrow = p.vb + n_ray * 128;
          uint32_t va[32], vb[32];
          ptx::tmem_ld_x32(t_lane + ch * 64, va);
          ptx::tmem_ld_x32(t_lane + ch * 64 + 32, vb);
          ptx::tmem_ld_wait();
          if (q == 0 && ch == 0 && lane < 8) write_bias_selector(sb + P2_ONES + X * 256, lane, 0, n_bias);   // next super-tile, layer 0
          ptx::tc_fence_before();
          ptx::fence_proxy_async_smem();
          arrive_leader(bar_act + 8 * X);                      // accumulator drained: next super-tile may start
          uint32_t mkv[2] = {0u, 0u};                             // EMIT: sign bits of this thread's 64 pre-activations
          // EMIT: post-ReLU fp16 copy of this thread's 64 columns = one row of K-block `ch` of the hv image, parked in K-block
          // 2 ch + 1 of the (dead) A tile -- this warp's own rows, drained by the l == D gate -- and copied out like the h_l slices
#pragma unroll
          for (int b = 0; b < 2; ++b) {
            const int col0 = ch * 64 + b * 32;
            const uint32_t (&v)[32] = b ? vb : va;
            const float4* vb4 = reinterpret_cast<const float4*>(vbrow + col0);
            const uint32_t w0 = a_heads + (uint32_t)(256 + col0) * 4u;
            uint32_t hh[4];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float4 bb = vb4[j];
              const float a0 = __uint_as_float(v[4 * j + 0]) + bb.x, a1 = __uint_as_float(v[4 * j + 1]) + bb.y;
              const float a2 = __uint_as_float(v[4 * j + 2]) + bb.z, a3 = __uint_as_float(v[4 * j + 3]) + bb.w;
              const float h0 = fmaxf(a0, 0.f), h1 = fmaxf(a1, 0.f), h2 = fmaxf(a2, 0.f), h3 = fmaxf(a3, 0.f);
              if (EMIT) {
                mkv[b] = mask_push(mask_push(mask_push(mask_push(mkv[b], a0), a1), a2), a3);
                hh[(j & 1) * 2] = ptx::cvt_f16x2(h0, h1); hh[(j & 1) * 2 + 1] = ptx::cvt_f16x2(h2, h3);
                if (j & 1) ptx::st_shared_v4(swk[b * 4 + (j >> 1)] + 16384u, hh[0], hh[1], hh[2], hh[3]);
              }
              const float4 wr = lds128(w0 + 16 * j), wg = lds128(w0 + 512 + 16 * j), wb = lds128(w0 + 1024 + 16 * j);
              hp0 = fmaf(h0, wr.x, hp0); hp0 = fmaf(h1, wr.y, hp0); hp0 = fmaf(h2, wr.z, hp0); hp0 = fmaf(h3, wr.w, hp0);
              hp1 = fmaf(h0, wg.x, hp1); hp1 = fmaf(h1, wg.y, hp1); hp1 = fmaf(h2, wg.z, hp1); hp1 = fmaf(h3, wg.w, hp1);
              hp2 = fmaf(h0, wb.x, hp2); hp2 = fmaf(h1, wb.y, hp2); hp2 = fmaf(h2, wb.z, hp2); hp2 = fmaf(h3, wb.w, hp2);
            }
          }
          if (EMIT) {
            *reinterpret_cast<uint2*>(mrec + (uint32_t)D * 4096u + (uint32_t)ch * 1024u + (uint32_t)r * 8u) = make_uint2(mkv[0], mkv[1]);
            emit_slice(arec + rec_act_hv(D), ch, 128, act_base + (uint32_t)(2 * ch + 1) * 16384u);
          }
        }
        if (l == defer_l && st > 0 && ch == 0) composite_st(st - 1);
      }
      // ---- heads: combine the two column halves -> raw (ch == 0 warps keep it for the deferred compositing) ----
      // the partials are parked in the first 2 KB of this slot's A tile, which is dead between the last layer's
      // d_full and the next super-tile's layer-0 epilogue (second barrier: nobody overwrites them before they are read)
      const uint32_t part = act_base + (uint32_t)r * 16u;
      if (ch == 1) sts128(part, make_float4(hp0, hp1, hp2, hp3));
      ptx::named_bar_sync(1 + X, 256);
      float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
      if (ch == 0) o = lds128(part);
      ptx::named_bar_sync(1 + X, 256);
      if (ch == 0) {
        if (p.use_viewdirs) pend = make_float4(hp0 + o.x + lds32(a_heads + 641 * 4), hp1 + o.y + lds32(a_heads + 642 * 4),
                                               hp2 + o.z + lds32(a_heads + 643 * 4), hp3 + o.w + lds32(a_heads + 640 * 4));
        else pend = make_float4(hp0 + o.x + lds32(a_heads + 1024 * 4), hp1 + o.y + lds32(a_heads + 1025 * 4),
                                hp2 + o.z + lds32(a_heads + 1026 * 4), hp3 + o.w + lds32(a_heads + 1027 * 4));
      }
    }
    if (ch == 0 && nst > 0) composite_st(nst - 1);                 // the last super-tile's rows
    if (EMIT && lane == 0) ptx::bulk_wait_all();
  } else {
    // =========================== sampler (warp 3) ===========================
    const int t = threadIdx.x - 96;                               // 0..31
    for (int st = 0; st < nst; ++st) {
      ptx::mbar_wait(bar_encfree, (st & 1) ^ 1);
      if (EMIT) { if (t == 0) ptx::bulk_wait_read0(); __syncwarp(); }   // the previous super-tile's encodings have been copied out
#pragma unroll 1
      for (int i = 0; i < 8; ++i) {
        const int X = i >> 2, tr_ = t + 32 * (i & 3);             // tile slot, tile row
        const int lr = st * TC_ST + X * TC_TILE + tr_;
        float px = 0.f, py = 0.f, pz = 0.f;
        if (lr < nrows) {
          const long long m = row_begin + lr;
          if (p.pts) { px = p.pts[m * 3]; py = p.pts[m * 3 + 1]; pz = p.pts[m * 3 + 2]; }
          else {
            const float* ry = p.rays + (ray0 + lr / p.S) * p.ray_stride;
            const float z = p.z_vals[m];
            px = __fadd_rn(ry[0], __fmul_rn(ry[3], z));                                       // run_nerf.py:381
            py = __fadd_rn(ry[1], __fmul_rn(ry[4], z));
            pz = __fadd_rn(ry[2], __fmul_rn(ry[5], z));
          }
        }
        encode_row_store(sb + SM_ENC + X * 16384 + act_row_off(tr_), tr_, px, py, pz, p.L);
      }
      ptx::fence_proxy_async_smem();
      arrive_leader(bar_encfull);
      if (EMIT && t == 0) {                                         // encodings of both slots -> their tile records
        for (int X = 0; X < 2; ++X)
          ptx::bulk_s2g(sv.act + (size_t)((blockIdx.x * sv.nst_plan + st) * 2 + X) * sv.rec_act, sb + SM_ENC + X * 16384, 16384u);
        ptx::bulk_commit();
      }
    }
    if (EMIT && t == 0) ptx::bulk_wait_all();
  }

  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync();                                  // the pair's MMAs / multicast commits are all done
  if (warp == 2) ptx::tmem_dealloc2(tmem, 512);
}

}  // namespace nb
