// fused_tc.cuh -- shared pieces of the fused tcgen05 network pass: shared-memory map, packed-weight layout and the
// packing kernels, the per-ray view-bias kernel, and the device helpers of the epilogue (swizzled A-tile stores,
// in-register positional encoding, segmented warp scans, the compositing of raw2outputs with its warp-to-warp carry).
//
// The pass itself -- pts = o + d*z -> positional encoding -> 8x256 MLP (+ heads) -> alpha compositing, replacing
// run_nerf.py:381-386 / :397-403 (run_network :37-51, batchify :27-34, Embedder.embed run_nerf_helpers.py:36-45,
// NeRF.forward :96-119, raw2outputs run_nerf.py:262-305) -- is march_tc2_kernel in fused_tc2.cuh (CTA pair,
// cta_group::2).  The single-CTA kernel it superseded lives in dev_kernels.cuh (libnerf_b200_dev.so only).
#pragma once
#include "common.cuh"
#include "tc_ptx.cuh"
#include "small_kernels.cuh"

namespace nb {

constexpr int TC_THREADS = 640;              // producer + issuer + spare + sampler warps, 16 epilogue warps
constexpr int TC_SAMPLER_THREADS = 32;       // (register allocation is per 4 warps: 20 warps x 96 regs fit)
constexpr int TC_W = 256;                 // hidden width supported by the tensor-core path
constexpr int TC_MAXD = 8;                // pts layers supported (bias table lives in smem)
constexpr int TC_TILE = 128;              // rows per MMA tile
constexpr int TC_ST = 256;                // rows per super-tile (two tile slots)
constexpr int TC_NST = 3;                 // weight ring stages
constexpr int TC_CHUNK_K = 32;            // K per weight chunk
constexpr uint32_t TC_STAGE_BYTES = 256 * TC_CHUNK_K * 2;   // 16 KB

// shared-memory map (bytes, relative to a 1024-aligned base)
constexpr uint32_t SM_ACT = 0;                                  // 2 x 64 KB  A operand (4 K-blocks x 16 KB)
constexpr uint32_t SM_ENC = 131072;                             // 2 x 16 KB  encoded inputs (1 K-block)
constexpr uint32_t SM_WRING = 163840;                           // 3 x 16 KB  weight ring
constexpr uint32_t SM_ONES = 212992;                            // 256 B: ONE 8-row atom of the bias-selector A slab (K=16, SWIZZLE_32B,
                                                                //        SBO = 0: all 128 rows read the same atom)
constexpr uint32_t SM_BIASB = SM_ONES + 512;                    // 213504: 8 KB resident B operand [256 x K=16]: all layers' biases
                                                                //        (one 256-byte selector atom per tile slot before it)
constexpr uint32_t SM_HEADS = SM_BIASB + 8192;                  // 221440: head weights, 4128 B
constexpr uint32_t SM_PART = SM_HEADS + 4128;                   // 225568: 2 x 128 x float4 partials
constexpr uint32_t SM_BARS = SM_PART + 4096;                    // mbarriers
constexpr uint32_t SM_MISC = SM_BARS + 256;                     // 229920: tmem ptr, compositing carry
constexpr uint32_t SM_TOTAL = SM_MISC + 128;                    // 230048
constexpr uint32_t SM_ALLOC = 230400 > SM_TOTAL ? 230400 : SM_TOTAL;                           // >= SM_TOTAL and the pair kernel's P2_TOTAL; dynamic smem base is 1024-aligned (checked at run time)
static_assert(SM_TOTAL <= SM_ALLOC, "shared-memory map exceeds the allocation");
constexpr uint32_t TC_BIAS_CHUNK_BYTES = 256 * 32;              // [256 rows x K=16] fp16: column pair (2l, 2l+1) = (hi, lo) of layer l's bias

// K columns of the resident bias operand used by bias layer `li` of `nb`: (hi, lo) pairs while 16 columns
// suffice, hi only for the last 2*nb-16 layers.  Returns hi column; *lo = lo column or -1.
__host__ __device__ inline int tc_bias_cols(int li, int nb, int* lo) {
  const int n_single = (2 * nb > 16) ? 2 * nb - 16 : 0, n_pair = nb - n_single;
  if (li < n_pair) { *lo = 2 * li + 1; return 2 * li; }
  *lo = -1;
  return 2 * n_pair + (li - n_pair);
}

// heads region (floats): viewdirs: alpha_w[256] rgb_w[3][128] alpha_b rgb_b[3]; else output_w[4][256] output_b[4]
constexpr int HEADS_FLOATS = 1032;

// ---------------------------------------------------------------------------------------------
// packed weight buffer
// ---------------------------------------------------------------------------------------------
struct PackLayout {
  int D, skip, use_viewdirs, IC, ICV, NL;
  int n_chunks;
  size_t off_chunks, chunk_bytes, off_bias, off_heads, off_vdir, off_biasb, off_pair, total;
  // backward (dgrad) stream: transposed weight chunks, linear image and its rank-split copy (bwd_tc2.cuh); 0 bytes when
  // the net has no view head (the tensor-core backward serves use_viewdirs nets)
  size_t off_bwd, bwd_bytes, off_bwd_pair;
};

__host__ __device__ inline int tc_layer_chunks(int l, int D, int skip) {
  if (l == 0) return 2;
  if (l < D && skip >= 0 && l == skip + 1) return 10;
  return 8;
}
__host__ __device__ inline uint32_t tc_layer_chunk_bytes(int l, int D) { return (l == D + 1) ? TC_STAGE_BYTES / 2 : TC_STAGE_BYTES; }
// every layer but the view layer (whose bias is per ray) starts with a bias chunk: one K=16 MMA of a
// constant-one A slab against [bias_hi, bias_lo, 0...] initialises the accumulator with the bias
__host__ __device__ inline bool tc_layer_has_bias(int l, int D) { return l != D + 1; }

static inline PackLayout make_pack_layout(const NerfNetParams& n) {
  PackLayout L;
  L.D = n.D; L.skip = n.skip; L.use_viewdirs = n.use_viewdirs; L.IC = n.input_ch; L.ICV = n.input_ch_views;
  L.NL = n.D + (n.use_viewdirs ? 2 : 0);
  L.n_chunks = 0; L.chunk_bytes = 0;
  for (int l = 0; l < L.NL; ++l) {
    int c = tc_layer_chunks(l, n.D, n.skip);
    L.n_chunks += c;
    L.chunk_bytes += (size_t)c * tc_layer_chunk_bytes(l, n.D);
  }
  L.off_chunks = 1024;
  L.off_bias = L.off_chunks + L.chunk_bytes;
  L.off_heads = L.off_bias + (size_t)(TC_MAXD + 1) * 1024;
  L.off_vdir = L.off_heads + HEADS_FLOATS * 4;
  L.off_biasb = L.off_vdir + (size_t)(128 * (n.input_ch_views > 0 ? n.input_ch_views : 1) + 128) * 4;
  L.off_biasb = (L.off_biasb + 255) & ~(size_t)255;
  L.off_pair = L.off_biasb + TC_BIAS_CHUNK_BYTES;          // rank-split copy of the chunk stream for the CTA-pair kernel
  L.off_bwd = L.off_pair + L.chunk_bytes;
  L.bwd_bytes = n.use_viewdirs ? (size_t)(4 + 8 * n.D) * TC_STAGE_BYTES : 0;
  L.off_bwd_pair = L.off_bwd + L.bwd_bytes;
  L.total = L.off_bwd_pair + L.bwd_bytes;
  return L;
}

// element (row n, k) of a chunk = src[n * sn + (k0 + k) * sk]: forward chunks read W[n][k0 + k] (sn = ld, sk = 1), the
// backward's transposed chunks read W[k0 + k][n] (sn = 1, sk = ld)
struct PackChunk { const float* src; int sn, sk, k0, kvalid, nrows; unsigned dst_off; };
constexpr int PACK_MAX_CHUNKS = 96;
struct PackJob { PackChunk c[PACK_MAX_CHUNKS]; int n; };

// one thread per 16-byte unit (8 fp16 of one row) of the swizzled chunk image
__global__ void pack_chunks_kernel(PackJob job, uint8_t* __restrict__ dst) {
  const int ci = blockIdx.y;
  if (ci >= job.n) return;
  const PackChunk c = job.c[ci];
  int u = blockIdx.x * blockDim.x + threadIdx.x;       // unit index: row * 4 + c16
  if (u >= c.nrows * 4) return;
  int row = u >> 2, c16 = u & 3;
  float v[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    int k = c16 * 8 + j;
    v[j] = (k < c.kvalid) ? c.src[(size_t)row * c.sn + (size_t)(c.k0 + k) * c.sk] : 0.0f;
  }
  uint4 o;
  o.x = ptx::cvt_f16x2(v[0], v[1]); o.y = ptx::cvt_f16x2(v[2], v[3]);
  o.z = ptx::cvt_f16x2(v[4], v[5]); o.w = ptx::cvt_f16x2(v[6], v[7]);
  // SWIZZLE_64B K-major: 8-row atoms of 512 B, 16B-chunk index ^= (row%8)>>1
  unsigned off = c.dst_off + (row >> 3) * 512 + (row & 7) * 64 + ((c16 ^ ((row & 7) >> 1)) << 4);
  *reinterpret_cast<uint4*>(dst + off) = o;
}

// resident bias operand: [256 rows x 16 K] fp16, K-major SWIZZLE_32B (rows of 32 B, 8-row atoms of 256 B)
struct PackBiasJob { const float* src[TC_MAXD + 2]; int n; unsigned dst_off; };
__global__ void pack_bias_kernel(PackBiasJob job, uint8_t* __restrict__ dst) {
  const int row = threadIdx.x;                         // 256 threads = 256 output rows
  __half h[16];
#pragma unroll
  for (int k = 0; k < 16; ++k) h[k] = __float2half_rn(0.0f);
  for (int li = 0; li < job.n; ++li) {
    const float b = job.src[li][row];
    int lo;
    const int hi = tc_bias_cols(li, job.n, &lo);
    const __half bh = __float2half_rn(b);
    h[hi] = bh;
    if (lo >= 0) h[lo] = __float2half_rn(b - __half2float(bh));
  }
  uint8_t* base = dst + job.dst_off + (row >> 3) * 256 + (row & 7) * 32;
  const int sw = ((row & 7) >> 2) & 1;                 // Swizzle<1,4,3>: 16-byte chunk index ^= bit 7 of the byte address
  uint4 c[2];
  for (int q = 0; q < 2; ++q) {
    const unsigned short* u = reinterpret_cast<const unsigned short*>(h + 8 * q);
    c[q] = make_uint4(u[0] | (u[1] << 16), u[2] | (u[3] << 16), u[4] | (u[5] << 16), u[6] | (u[7] << 16));
  }
  *reinterpret_cast<uint4*>(base + ((0 ^ sw) << 4)) = c[0];
  *reinterpret_cast<uint4*>(base + ((1 ^ sw) << 4)) = c[1];
}

struct PackTables { NerfNetParams net; size_t off_bias, off_heads, off_vdir; };
__global__ void pack_tables_kernel(PackTables t, uint8_t* __restrict__ dst) {
  const NerfNetParams& n = t.net;
  float* bias = reinterpret_cast<float*>(dst + t.off_bias);
  float* heads = reinterpret_cast<float*>(dst + t.off_heads);
  float* vdir = reinterpret_cast<float*>(dst + t.off_vdir);
  const int tid = blockIdx.x * blockDim.x + threadIdx.x, nt = gridDim.x * blockDim.x;
  for (int i = tid; i < (TC_MAXD + 1) * 256; i += nt) {
    int l = i >> 8, c = i & 255;
    float v = 0.0f;
    if (l < n.D) v = n.pts_b[l][c];
    else if (l == n.D && n.use_viewdirs) v = n.feature_b[c];
    bias[i] = v;
  }
  if (n.use_viewdirs) {
    for (int i = tid; i < 256; i += nt) heads[i] = n.alpha_w[i];
    for (int i = tid; i < 384; i += nt) heads[256 + i] = n.rgb_w[i];
    if (tid == 0) { heads[640] = n.alpha_b[0]; heads[641] = n.rgb_b[0]; heads[642] = n.rgb_b[1]; heads[643] = n.rgb_b[2]; }
    const int ICV = n.input_ch_views;
    for (int i = tid; i < 128 * ICV; i += nt) { int j = i / ICV, c = i % ICV; vdir[i] = n.views_w[(size_t)j * (256 + ICV) + 256 + c]; }
    for (int i = tid; i < 128; i += nt) vdir[128 * ICV + i] = n.views_b[i];
  } else {
    for (int i = tid; i < 1024; i += nt) heads[i] = n.output_w[i];        // first 4 rows of output_linear
    for (int i = tid; i < 4; i += nt) heads[1024 + i] = n.output_b[i];
  }
}

// view-direction contribution of views_linears[0], once per ray (the reference recomputes it per
// sample through the expand at run_nerf.py:44-46):  vb[n][j] = b[j] + sum_c W[j][256+c] * enc(v_n)[c]
constexpr int VB_RAYS = 8;        // rays per block (512 blocks for a 4096-ray chunk: the kernel is latency-bound)
__global__ void __launch_bounds__(128) view_bias_kernel(const float* __restrict__ dirs, int dir_stride, long long N, int Lv, int ICV,
                                                     const float* __restrict__ vdir, float* __restrict__ vb) {
  __shared__ float s_enc[VB_RAYS][64];
  const long long n0 = (long long)blockIdx.x * VB_RAYS;
  const int j = threadIdx.x;
  for (int i = threadIdx.x; i < VB_RAYS * ICV; i += 128) {
    const int r = i / ICV, c = i - r * ICV;
    float v = 0.0f;
    if (n0 + r < N) {
      const float* d = dirs + (n0 + r) * dir_stride;
      if (c < 3) v = d[c];
      else { int f = (c - 3) / 6, q = (c - 3) % 6; float a = __fmul_rn(d[q % 3], exp2f((float)f)); v = (q < 3) ? sinf(a) : cosf(a); }
    }
    s_enc[r][c] = v;
  }
  float w[64];
#pragma unroll
  for (int c = 0; c < 64; ++c) w[c] = (c < ICV) ? vdir[j * ICV + c] : 0.0f;
  const float b = vdir[128 * ICV + j];
  __syncthreads();
  for (int r = 0; r < VB_RAYS && n0 + r < N; ++r) {
    float acc = b;
#pragma unroll
    for (int c = 0; c < 64; ++c) if (c < ICV) acc = fmaf(w[c], s_enc[r][c], acc);
    vb[(n0 + r) * 128 + j] = acc;
  }
}

// One launch per ray chunk for everything the two fused passes need per RAY (render_rays' prologue, run_nerf.py:351-379 and
// the per-ray part of run_network, :44-46): the coarse z row (as coarse_z_kernel) and the view-bias rows of BOTH networks
// (as view_bias_kernel) -- three launches of round 1 folded into one, and the fine net's table is off the critical path
// between the resampling and the fine pass.  256 threads: threads 0-127 serve net A's 128 view units, 128-255 net B's.
struct RaySetupArgs {
  const float* rays; int ray_stride; long long N; int Lv, ICV;
  const float* vdir_a; float* vb_a;               // net A side table (128 x ICV weights + 128 biases) -> vb_a [N,128]
  const float* vdir_b; float* vb_b;               // net B or NULL
  const float* t_vals; const float* t_rand; int S, lindisp; float* z_out;   // z_out NULL: no z sampling
  float* pack_out;                                // not NULL: the block first BUILDS its rows of `rays` (render()'s ray batch
  PackRaysArgs pack;                              //           construction, pack_ray_row) -- same buffer as `rays`
};
__device__ __forceinline__ float setup_z_at(float near, float far, float t, int lindisp) {
  const float omt = __fsub_rn(1.0f, t);
  if (!lindisp) return __fadd_rn(__fmul_rn(near, omt), __fmul_rn(far, t));                    // run_nerf.py:359
  const float a = __fmul_rn(__fdiv_rn(1.0f, near), omt), b = __fmul_rn(__fdiv_rn(1.0f, far), t);
  return __fdiv_rn(1.0f, __fadd_rn(a, b));                                                     // :361
}
__global__ void __launch_bounds__(256) ray_setup_kernel(const RaySetupArgs a) {
  __shared__ float s_enc[VB_RAYS][64];
  const long long n0 = (long long)blockIdx.x * VB_RAYS;
  const int j = threadIdx.x & 127, net = threadIdx.x >> 7;
  const int ICV = a.ICV;
  if (a.pack_out != nullptr) {                      // run_nerf.py:95-123 for this block's rays, then everyone reads them back
    if (threadIdx.x < VB_RAYS && n0 + threadIdx.x < a.N) pack_ray_row(a.pack, n0 + threadIdx.x, a.pack_out);
    __syncthreads();
  }
  if (a.vb_a != nullptr) {
    for (int i = threadIdx.x; i < VB_RAYS * ICV; i += 256) {
      const int r = i / ICV, c = i - r * ICV;
      float v = 0.0f;
      if (n0 + r < a.N) {
        const float* d = a.rays + (n0 + r) * a.ray_stride + 8;
        if (c < 3) v = d[c];
        else { const int f = (c - 3) / 6, q = (c - 3) % 6; const float x = __fmul_rn(d[q % 3], exp2f((float)f)); v = (q < 3) ? sinf(x) : cosf(x); }
      }
      s_enc[r][c] = v;
    }
    const float* vdir = net ? a.vdir_b : a.vdir_a;
    float* vb = net ? a.vb_b : a.vb_a;
    float w[64];
    float b = 0.f;
    if (vdir != nullptr) {
#pragma unroll
      for (int c = 0; c < 64; ++c) w[c] = (c < ICV) ? vdir[j * ICV + c] : 0.0f;
      b = vdir[128 * ICV + j];
    }
    __syncthreads();
    if (vdir != nullptr) {
      for (int r = 0; r < VB_RAYS && n0 + r < a.N; ++r) {
        float acc = b;
#pragma unroll
        for (int c = 0; c < 64; ++c) if (c < ICV) acc = fmaf(w[c], s_enc[r][c], acc);
        vb[(n0 + r) * 128 + j] = acc;
      }
    }
  }
  if (a.z_out != nullptr) {                          // z sampling of the block's rays (coarse_z_kernel's arithmetic)
    for (int i = threadIdx.x; i < VB_RAYS * a.S; i += 256) {
      const int r = i / a.S, s = i - r * a.S;
      const long long n = n0 + r;
      if (n >= a.N) break;
      const float near = a.rays[n * a.ray_stride + 6], far = a.rays[n * a.ray_stride + 7];
      float z = setup_z_at(near, far, a.t_vals[s], a.lindisp);
      if (a.t_rand != nullptr) {
        const float zl = (s > 0) ? setup_z_at(near, far, a.t_vals[s - 1], a.lindisp) : z;
        const float zu = (s < a.S - 1) ? setup_z_at(near, far, a.t_vals[s + 1], a.lindisp) : z;
        const float lower = (s > 0) ? __fmul_rn(0.5f, __fadd_rn(z, zl)) : z;                    // :367-369
        const float upper = (s < a.S - 1) ? __fmul_rn(0.5f, __fadd_rn(zu, z)) : z;
        z = __fadd_rn(lower, __fmul_rn(__fsub_rn(upper, lower), a.t_rand[n * a.S + s]));        // :379
      }
      a.z_out[n * a.S + s] = z;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// fused march kernel
// ---------------------------------------------------------------------------------------------
struct MarchParams {
  const float* rays; int ray_stride;      // [N, ray_stride]  (o,d,near,far[,viewdir]) or NULL in pts mode
  const float* z_vals;                    // [N,S]
  const float* pts;                       // [N*S,3] (pts mode: run_network) or NULL
  const float* noise;                     // [N,S] or NULL
  const float* vb;                        // [N,128] view bias (use_viewdirs)
  long long N; int S; int rays_per_cta;
  const uint8_t* chunks; const float* bias; const float* heads; const uint8_t* biasb;
  int D, skip, use_viewdirs, L, IC;
  int white_bkgd, do_composite;
  NerfPassOut out;
  unsigned long long pair_half_bytes;     // pair kernel: bytes of one rank's half of the chunk stream
};

// compositing carry of the ray that is still open at a warp boundary (shared memory, 32 B)
constexpr uint32_t CARRY_T = 0, CARRY_R = 4, CARRY_G = 8, CARRY_B = 12, CARRY_D = 16, CARRY_A = 20, CARRY_TURN = 24;

__device__ __forceinline__ uint32_t act_row_off(int r) { return (uint32_t)((r >> 3) * 1024 + (r & 7) * 128); }

__device__ __forceinline__ float4 lds128(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ float lds32(uint32_t addr) { float v; asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr)); return v; }
__device__ __forceinline__ void sts32(uint32_t addr, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory"); }
__device__ __forceinline__ void sts128(uint32_t addr, float4 v) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_shared(uint32_t addr) {
  uint32_t v; asm volatile("ld.acquire.cta.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory"); return v;
}
__device__ __forceinline__ void st_release_shared(uint32_t addr, uint32_t v) {
  asm volatile("st.release.cta.shared.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}
// (a, b) += (c, d) as one packed FADD2
__device__ __forceinline__ void add2(float& a, float& b, float c, float d) {
  asm("{\n\t.reg .b64 ra, rb, rc;\n\tmov.b64 ra, {%0, %1};\n\tmov.b64 rb, {%2, %3};\n\tadd.rn.f32x2 rc, ra, rb;\n\tmov.b64 {%0, %1}, rc;\n\t}"
      : "+f"(a), "+f"(b) : "f"(c), "f"(d));
}

// v[32] (fp32 accumulators of one row, bias already added) -> (ReLU) -> fp16 -> 4 x 16-byte stores
// into the 128B-swizzled K-major A tile.
template <bool RELU>
__device__ __forceinline__ void store_act32(const float (&x)[32], uint32_t act_base, int r, int col0) {
  const uint32_t kb = (uint32_t)(col0 >> 6) * 16384u;
  const int c16_0 = (col0 & 63) >> 3;
  const uint32_t row = act_base + kb + act_row_off(r);
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    uint32_t h0, h1, h2, h3;
    if (RELU) {
      h0 = ptx::cvt_relu_f16x2(x[g * 8 + 0], x[g * 8 + 1]); h1 = ptx::cvt_relu_f16x2(x[g * 8 + 2], x[g * 8 + 3]);
      h2 = ptx::cvt_relu_f16x2(x[g * 8 + 4], x[g * 8 + 5]); h3 = ptx::cvt_relu_f16x2(x[g * 8 + 6], x[g * 8 + 7]);
    } else {
      h0 = ptx::cvt_f16x2(x[g * 8 + 0], x[g * 8 + 1]); h1 = ptx::cvt_f16x2(x[g * 8 + 2], x[g * 8 + 3]);
      h2 = ptx::cvt_f16x2(x[g * 8 + 4], x[g * 8 + 5]); h3 = ptx::cvt_f16x2(x[g * 8 + 6], x[g * 8 + 7]);
    }
    ptx::st_shared_v4(row + (uint32_t)(((c16_0 + g) ^ (r & 7)) << 4), h0, h1, h2, h3);
  }
}

// Same, with the 8 swizzled 16-byte-chunk addresses of this thread's row precomputed once
// (sw[c] = tile base + row offset + ((c ^ (r & 7)) << 4)): every store is [register + immediate].
template <bool RELU, int COL0>
__device__ __forceinline__ void store_act32_pre(const float (&x)[32], const uint32_t (&sw)[8]) {
  constexpr uint32_t kb = (uint32_t)(COL0 >> 6) * 16384u;
  constexpr int c16_0 = (COL0 & 63) >> 3;
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    uint32_t h0, h1, h2, h3;
    if (RELU) {
      h0 = ptx::cvt_relu_f16x2(x[g * 8 + 0], x[g * 8 + 1]); h1 = ptx::cvt_relu_f16x2(x[g * 8 + 2], x[g * 8 + 3]);
      h2 = ptx::cvt_relu_f16x2(x[g * 8 + 4], x[g * 8 + 5]); h3 = ptx::cvt_relu_f16x2(x[g * 8 + 6], x[g * 8 + 7]);
    } else {
      h0 = ptx::cvt_f16x2(x[g * 8 + 0], x[g * 8 + 1]); h1 = ptx::cvt_f16x2(x[g * 8 + 2], x[g * 8 + 3]);
      h2 = ptx::cvt_f16x2(x[g * 8 + 4], x[g * 8 + 5]); h3 = ptx::cvt_f16x2(x[g * 8 + 6], x[g * 8 + 7]);
    }
    ptx::st_shared_v4(sw[c16_0 + g] + kb, h0, h1, h2, h3);
  }
}

// segmented (per-ray) inclusive scans over one warp; `s` = lane of the segment start at or before
// this lane inside the warp, or -1 when the segment began in an earlier warp.
__device__ __forceinline__ float seg_scan_mul(float v, int lane, int s) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { float t = __shfl_up_sync(0xffffffffu, v, o); if (lane >= o && lane - o >= s) v *= t; }
  return v;
}
__device__ __forceinline__ float seg_scan_add(float v, int lane, int s) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { float t = __shfl_up_sync(0xffffffffu, v, o); if (lane >= o && lane - o >= s) v += t; }
  return v;
}

// One 32-column batch of a hidden-layer epilogue: the bias is already in the accumulator (bias chunk)
__device__ __forceinline__ void as_float32(const uint32_t (&v)[32], float (&x)[32]) {
#pragma unroll
  for (int j = 0; j < 32; ++j) x[j] = __uint_as_float(v[j]);
}

// Row `r` (0..7) of the 8-row bias-selector A atom for bias layer `li`: 1.0 in that layer's K columns.
__device__ __forceinline__ void write_bias_selector(uint32_t slab, int r, int li, int nb) {
  int lo;
  const int hi = tc_bias_cols(li, nb, &lo);
  uint32_t w[8] = {0, 0, 0, 0, 0, 0, 0, 0};            // 16 halves as 8 words
  w[hi >> 1] |= (hi & 1) ? 0x3c000000u : 0x00003c00u;
  if (lo >= 0) w[lo >> 1] |= (lo & 1) ? 0x3c000000u : 0x00003c00u;
  const int sw = (r >> 2) & 1;
  const uint32_t a = slab + (uint32_t)(r * 32);
  ptx::st_shared_v4(a + ((0 ^ sw) << 4), w[0], w[1], w[2], w[3]);
  ptx::st_shared_v4(a + ((1 ^ sw) << 4), w[4], w[5], w[6], w[7]);
}

// Positional encoding of one point into its 128-byte K-block row of the A operand (64 fp16 channels:
// x y z, then per frequency sin(2^f xyz), cos(2^f xyz); channel 63 is zero padding), written as eight
// 16-byte swizzled chunks.  run_nerf_helpers.py:36-45 evaluates sin/cos of 2^f x for every f; here only
// f = 0 and f = 5 are evaluated with sincosf, the other octaves come from the double-angle identities
// sin 2a = 2 sin a cos a, cos 2a = (cos a - sin a)(cos a + sin a).  Four doublings amplify the fp32
// rounding of the anchor to <= 1.6e-6 absolute (numpy model over [-6, 6]: 0.07 % of the fp16 operand
// values move by one fp16 ulp), far below the fp16 quantisation of the operand itself, and cut the
// sampler warp's work ~4x: with 30 sincosf per row it took longer than the MMAs of half a super-tile and
// the issuers idled on enc_full (profiles/r01_summary.md, "sampler").
__device__ __forceinline__ void encode_row_store(uint32_t row, int tr_, float px, float py, float pz, int L) {
  uint32_t h[32];
  float s[3], c[3];
  const float q[3] = {px, py, pz};
  float carry = 0.f;                                   // pending even-indexed channel of the current pair
  int n = 0;                                           // channels emitted so far (compile-time after unrolling)
  auto emit = [&](float v) {
    if (n & 1) { __half2 hh = __floats2half2_rn(carry, v); h[n >> 1] = *reinterpret_cast<uint32_t*>(&hh); }
    else carry = v;
    ++n;
  };
  emit(px); emit(py); emit(pz);
#pragma unroll
  for (int f = 0; f < 10; ++f) {
    if (f == 0 || f == 5) {
#pragma unroll
      for (int j = 0; j < 3; ++j) sincosf(q[j] * (float)(1 << f), &s[j], &c[j]);
    } else {
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        const float s2 = (s[j] + s[j]) * c[j], c2 = (c[j] - s[j]) * (c[j] + s[j]);
        s[j] = s2; c[j] = c2;
      }
    }
    const bool on = f < L;
#pragma unroll
    for (int j = 0; j < 3; ++j) emit(on ? s[j] : 0.f);
#pragma unroll
    for (int j = 0; j < 3; ++j) emit(on ? c[j] : 0.f);
  }
  emit(0.f);
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const uint32_t a = row + (uint32_t)((k ^ (tr_ & 7)) << 4);
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(h[4 * k]), "r"(h[4 * k + 1]), "r"(h[4 * k + 2]), "r"(h[4 * k + 3]) : "memory");
  }
}

// raw (rgb, sigma) of one row per lane -> alpha compositing of whole rays (run_nerf.py:275-303) with the carry of the
// ray that is open at the warp boundary threaded warp -> warp through shared memory (ticket order: st, slot, q).
__device__ __forceinline__ void composite_rows(const MarchParams& p, const float4 raw4, const bool valid, const int lr, const int rl,
                                               const long long n_ray, const long long row_begin, const int st, const int X,
                                               const int q, const int lane, const uint32_t a_carry) {
  const long long m = row_begin + lr;
  if (valid && p.out.raw) reinterpret_cast<float4*>(p.out.raw)[m] = raw4;
  if (!p.do_composite) return;
  const int k = lr - rl * p.S;
  float alpha = 0.f, cr = 0.f, cg = 0.f, cb = 0.f, z = 0.f;
  if (valid) {
    const float* rd = p.rays + n_ray * p.ray_stride + 3;
    const float norm = sqrtf(rd[0] * rd[0] + rd[1] * rd[1] + rd[2] * rd[2]);         // run_nerf.py:280
    z = p.z_vals[m];
    float dist = (k == p.S - 1) ? 1e10f : __fsub_rn(p.z_vals[m + 1], z);             // :277-278
    dist = __fmul_rn(dist, norm);
    const float sg = raw4.w + (p.noise ? p.noise[m] : 0.0f);
    alpha = __fsub_rn(1.0f, expf(-fmaxf(sg, 0.0f) * dist));                           // :275
    cr = sigmoidf_acc(raw4.x); cg = sigmoidf_acc(raw4.y); cb = sigmoidf_acc(raw4.z); // :282
  }
  const bool seg_start = valid && (k == 0), seg_end = valid && (k == p.S - 1);
  const unsigned smask = __ballot_sync(0xffffffffu, seg_start);
  const unsigned below = smask & ((lane == 31) ? 0xffffffffu : ((2u << lane) - 1u));
  const int s = below ? (31 - __clz(below)) : -1;
  const float qv = valid ? __fadd_rn(__fsub_rn(1.0f, alpha), 1e-10f) : 1.0f;         // :295
  const float pv = seg_scan_mul(qv, lane, s);
  float ev = __shfl_up_sync(0xffffffffu, pv, 1);
  if (lane == 0 || s == lane) ev = 1.0f;
  const float wl = valid ? alpha * ev : 0.0f;
  float t_r = seg_scan_add(wl * cr, lane, s), t_g = seg_scan_add(wl * cg, lane, s), t_b = seg_scan_add(wl * cb, lane, s);
  float t_d = seg_scan_add(wl * z, lane, s), t_a = seg_scan_add(wl, lane, s);
  const uint32_t ticket = (uint32_t)((st * 2 + X) * 4 + q);
  if (lane == 0) { while (ld_acquire_shared(a_carry + CARRY_TURN) != ticket) { } }
  __syncwarp();
  const float Tin = lds32(a_carry + CARRY_T);
  const float c_r = lds32(a_carry + CARRY_R), c_g = lds32(a_carry + CARRY_G), c_b = lds32(a_carry + CARRY_B);
  const float c_d = lds32(a_carry + CARRY_D), c_a = lds32(a_carry + CARRY_A);
  __syncwarp();
  if (s < 0) { t_r = fmaf(Tin, t_r, c_r); t_g = fmaf(Tin, t_g, c_g); t_b = fmaf(Tin, t_b, c_b); t_d = fmaf(Tin, t_d, c_d); t_a = fmaf(Tin, t_a, c_a); }
  if (lane == 31) {
    if (seg_end) {
      sts32(a_carry + CARRY_T, 1.0f); sts32(a_carry + CARRY_R, 0.f); sts32(a_carry + CARRY_G, 0.f); sts32(a_carry + CARRY_B, 0.f);
      sts32(a_carry + CARRY_D, 0.f); sts32(a_carry + CARRY_A, 0.f);
    } else {
      sts32(a_carry + CARRY_T, (s >= 0) ? pv : Tin * pv);
      sts32(a_carry + CARRY_R, t_r); sts32(a_carry + CARRY_G, t_g); sts32(a_carry + CARRY_B, t_b);
      sts32(a_carry + CARRY_D, t_d); sts32(a_carry + CARRY_A, t_a);
    }
    st_release_shared(a_carry + CARRY_TURN, ticket + 1u);
  }
  if (valid && p.out.weights) p.out.weights[m] = (s < 0) ? Tin * wl : wl;
  if (seg_end) {
    float rr = t_r, gg = t_g, bb = t_b;
    if (p.white_bkgd) { const float bg = 1.0f - t_a; rr += bg; gg += bg; bb += bg; }  // :302-303
    if (p.out.rgb_map) { p.out.rgb_map[n_ray * 3] = rr; p.out.rgb_map[n_ray * 3 + 1] = gg; p.out.rgb_map[n_ray * 3 + 2] = bb; }
    if (p.out.disp_map) {
      const float ratio = t_d / t_a;
      const float mm = (ratio != ratio) ? ratio : fmaxf(1e-10f, ratio);              // :299
      p.out.disp_map[n_ray] = 1.0f / mm;
    }
    if (p.out.acc_map) p.out.acc_map[n_ray] = t_a;
    if (p.out.depth_map) p.out.depth_map[n_ray] = t_d;
  }
}

extern __shared__ __align__(1024) uint8_t tc_smem[];

}  // namespace nb
