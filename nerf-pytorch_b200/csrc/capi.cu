// capi.cu -- extern "C" entry points of libnerf_b200.so (see include/nerf_b200.h).
#include <stdarg.h>
#include "common.cuh"
#include "small_kernels.cuh"
#include "bwd_simt.cuh"
#include "mlp_simt.cuh"
#include "fused_tc.cuh"
#include "fused_tc2.cuh"
#include "bwd_tc2.cuh"
#include "train_step.cuh"

namespace nb {
thread_local char g_err[512] = {0};
long long g_launches = 0;
int set_error(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

// ---- optional device-time accounting of march_tc_kernel launches (bench.py roofline) ----
struct TimedLaunch { cudaEvent_t a, b; double flops; int kind; };   // kind 0: forward pass, 1: dgrad chain, 2: wgrad
static bool g_timing = false;
static TimedLaunch g_timed[4096];
static int g_ntimed = 0;

static double net_macs_per_row(const NerfNetParams& n) {
  // MACs of the reference's Linear layers per sample row (SURVEY Appendix B)
  double m = (double)n.input_ch * n.W;
  for (int i = 1; i < n.D; ++i) m += (double)((n.skip >= 0 && i == n.skip + 1) ? n.W + n.input_ch : n.W) * n.W;
  if (n.use_viewdirs) m += (double)n.W * n.W + n.W + (double)(n.W + n.input_ch_views) * (n.W / 2) + 3.0 * (n.W / 2);
  else m += (double)n.W * n.output_ch;
  return m;
}

static int check_tc_net(const NerfNetParams* net) {
  NB_CHECK_ARG(net != nullptr, "net is NULL");
  NB_CHECK_ARG(net->W == TC_W, "tensor-core path supports netwidth == 256 (got %d); use precision=FP32", net->W);
  NB_CHECK_ARG(net->D >= 2 && net->D <= TC_MAXD, "tensor-core path supports 2 <= netdepth <= %d (got %d)", TC_MAXD, net->D);
  NB_CHECK_ARG(net->input_ch >= 3 && net->input_ch <= 63, "input_ch must be in [3,63] (got %d)", net->input_ch);
  NB_CHECK_ARG(net->skip < net->D - 1, "skip layer must be < D-1");
  if (net->use_viewdirs) NB_CHECK_ARG(net->input_ch_views >= 3 && net->input_ch_views <= 63, "input_ch_views must be in [3,63]");
  return 0;
}

static int smem_optin(const void* fn, size_t bytes) {
  NB_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  return 0;
}

// per-device facts (SM count; which kernels already have their > 48 KB shared-memory opt-in): the library may be used
// on several devices of one process, and cudaFuncSetAttribute is per device
struct DeviceState { int sms; bool optin_fwd, optin_bwd; cudaStream_t side; cudaEvent_t ev[4]; };
static DeviceState* device_state() {
  static DeviceState st[64];
  static bool init[64] = {false};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64) dev = 0;
  if (!init[dev]) {
    int n = 0;
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    st[dev].sms = n > 0 ? n : 148;
    st[dev].optin_fwd = st[dev].optin_bwd = false;
    // side stream + events of the two-pass backward: created with the device state (the first library call on a device), not
    // lazily inside a call that may be running under stream capture
    st[dev].side = nullptr;
    if (cudaStreamCreateWithFlags(&st[dev].side, cudaStreamNonBlocking) == cudaSuccess) {
      for (int i = 0; i < 4; ++i)
        if (cudaEventCreateWithFlags(&st[dev].ev[i], cudaEventDisableTiming) != cudaSuccess) { cudaStreamDestroy(st[dev].side); st[dev].side = nullptr; break; }
    } else {
      st[dev].side = nullptr;
    }
    cudaGetLastError();
    init[dev] = true;
  }
  return &st[dev];
}
static int num_sms() { return device_state()->sms; }

typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                             const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                             CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
// 2-D tensor map over a byte buffer viewed as [rows][256] uint16 (512-byte rows); box = `box_rows` rows (box_rows * 512 bytes)
static int make_row_map(CUtensorMap* map, const void* base, size_t bytes, int box_rows) {
  static EncodeFn encode = nullptr;
  if (!encode) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    NB_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
    NB_CHECK_ARG(fn != nullptr && qres == cudaDriverEntryPointSuccess, "cuTensorMapEncodeTiled not available");
    encode = reinterpret_cast<EncodeFn>(fn);
  }
  NB_CHECK_ARG(bytes % 512 == 0 && (reinterpret_cast<uintptr_t>(base) & 15) == 0, "tensor map: buffer must be 16-byte aligned, a multiple of 512 bytes");
  const cuuint64_t gdim[2] = {256, (cuuint64_t)(bytes / 512)};
  const cuuint64_t gstr[1] = {512};
  const cuuint32_t box[2] = {256, (cuuint32_t)box_rows}, estr[2] = {1, 1};
  CUresult cr = encode(map, CU_TENSOR_MAP_DATA_TYPE_UINT16, 2, const_cast<void*>(base), gdim, gstr, box, estr,
                       CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                       CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  NB_CHECK_ARG(cr == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed (%d)", (int)cr);
  return 0;
}

// shared launcher of the fused tcgen05 pass; `save` != NULL selects the training-mode kernel (EMIT)
static int launch_march(const float* rays, int ray_stride, const float* z_vals, const float* pts,
                        const float* dirs, int dir_stride, const float* noise, long long N, int S,
                        const NerfNetParams* net, const void* packed, int L, int Lv, int white_bkgd, int do_composite,
                        const NerfPassOut* out, void* workspace, size_t workspace_bytes, const NerfTrainSave* save, const float* vb_pre,
                        cudaStream_t st) {
  if (int rc = check_tc_net(net)) return rc;
  NB_CHECK_ARG(packed != nullptr, "packed weights are NULL (call nerf_b200_pack_weights)");
  NB_CHECK_ARG(N > 0 && S > 0, "empty ray batch must be handled by the caller (N=%lld S=%d)", N, S);
  NB_CHECK_ARG((long long)N * S < (1ll << 40), "batch too large");
  NB_CHECK_ARG(3 + 6 * L == net->input_ch || (L == 0 && net->input_ch == 3), "multires %d does not match input_ch %d", L, net->input_ch);
  const PackLayout PL = make_pack_layout(*net);
  const uint8_t* pk = static_cast<const uint8_t*>(packed);
  MarchParams p;
  memset(&p, 0, sizeof(p));
  p.rays = rays; p.ray_stride = ray_stride; p.z_vals = z_vals; p.pts = pts; p.noise = noise;
  p.N = N; p.S = S;
  p.bias = reinterpret_cast<const float*>(pk + PL.off_bias);
  p.heads = reinterpret_cast<const float*>(pk + PL.off_heads);
  p.biasb = pk + PL.off_biasb;
  p.D = net->D; p.skip = net->skip; p.use_viewdirs = net->use_viewdirs; p.L = L; p.IC = net->input_ch;
  p.white_bkgd = white_bkgd; p.do_composite = do_composite;
  if (out) p.out = *out;
  if (net->use_viewdirs && vb_pre != nullptr) {
    p.vb = vb_pre;                                     // the per-ray view-bias table was prepared by ray_setup_kernel
  } else if (net->use_viewdirs) {
    NB_CHECK_ARG(dirs != nullptr, "viewdirs required by a use_viewdirs network");
    NB_CHECK_ARG(workspace != nullptr && workspace_bytes >= (size_t)N * 128 * 4, "workspace too small: need %zu bytes", (size_t)N * 128 * 4);
    NB_CHECK_ARG(3 + 6 * Lv == net->input_ch_views || (Lv == 0 && net->input_ch_views == 3), "multires_views mismatch");
    float* vb = static_cast<float*>(workspace);
    view_bias_kernel<<<cdiv(N, VB_RAYS), 128, 0, st>>>(dirs, dir_stride, N, Lv, net->input_ch_views,
                                                  reinterpret_cast<const float*>(pk + PL.off_vdir), vb);
    NB_LAUNCH_OK("view_bias_kernel");
    p.vb = vb;
  }
  // persistent grid: whole rays per CTA, balanced over the SMs, whole CTA pairs (a padding CTA owns no rays)
  DeviceState* ds = device_state();
  const TilePlan plan = make_tile_plan(N, S, ds->sms);
  p.rays_per_cta = plan.rays_per_cta;
  NB_CHECK_ARG((long long)p.rays_per_cta * S < (1ll << 30), "rays_per_cta * S overflows");
  if (!ds->optin_fwd) {
    if (int rc = smem_optin((const void*)march_tc2_kernel<false>, SM_ALLOC)) return rc;
    if (int rc = smem_optin((const void*)march_tc2_kernel<true>, SM_ALLOC)) return rc;
    ds->optin_fwd = true;
  }
  TrainSaveDev sv;
  memset(&sv, 0, sizeof(sv));
  if (save) {
    NB_CHECK_ARG(net->use_viewdirs, "training-mode records are implemented for use_viewdirs networks");
    NB_CHECK_ARG(save->act && save->mask, "training-mode save buffers are NULL");
    NB_CHECK_ARG(save->act_bytes >= (size_t)plan.n_tiles * rec_act_bytes(net->D) && save->mask_bytes >= (size_t)plan.n_tiles * rec_mask_bytes(net->D),
                 "training-mode save buffers too small (see nerf_b200_train_record_bytes)");
    NB_CHECK_ARG((reinterpret_cast<uintptr_t>(save->act) & 15) == 0 && (reinterpret_cast<uintptr_t>(save->mask) & 15) == 0, "save buffers must be 16-byte aligned");
    sv.act = static_cast<uint8_t*>(save->act); sv.mask = static_cast<uint8_t*>(save->mask);
    sv.nst_plan = plan.nst; sv.rec_act = rec_act_bytes(net->D); sv.rec_mask = rec_mask_bytes(net->D);
  }
  TimedLaunch* tl = nullptr;
  if (g_timing && g_ntimed < 4096) {
    tl = &g_timed[g_ntimed++];
    cudaEventCreate(&tl->a); cudaEventCreate(&tl->b);
    tl->flops = 2.0 * net_macs_per_row(*net) * (double)(N * (long long)S);
    tl->kind = 0;
    cudaEventRecord(tl->a, st);
  }
  // tensor map over the rank-split chunk stream (512-byte rows); box = 16 rows = 8 KB = one ring stage
  CUtensorMap wmap;
  const uint8_t* pair_stream = pk + PL.off_pair;
  p.chunks = pair_stream;
  p.pair_half_bytes = PL.chunk_bytes / 2;
  if (int rc = make_row_map(&wmap, pair_stream, PL.chunk_bytes, 16)) return rc;
  if (save) march_tc2_kernel<true><<<plan.grid, TC_THREADS, SM_ALLOC, st>>>(p, wmap, sv);
  else march_tc2_kernel<false><<<plan.grid, TC_THREADS, SM_ALLOC, st>>>(p, wmap, sv);
  if (tl) cudaEventRecord(tl->b, st);
  NB_LAUNCH_OK("march_tc2_kernel");
  return 0;
}

}  // namespace nb

using namespace nb;

extern "C" {

int nerf_b200_abi_version(void) { return NERF_B200_ABI_VERSION; }
const char* nerf_b200_last_error(void) { return g_err; }
int64_t nerf_b200_launch_count(void) { return g_launches; }

int nerf_b200_timing_enable(int on) { g_timing = on != 0; return 0; }
int nerf_b200_timing_read(double* kernel_ms, int64_t* launches, double* algorithmic_flops) {
  return nerf_b200_timing_read_kinds(kernel_ms, launches, algorithmic_flops, nullptr);
}
// kind_ms[3]: device time of the forward passes, the dgrad chains and the wgrad kernels (NULL: not wanted)
int nerf_b200_timing_read_kinds(double* kernel_ms, int64_t* launches, double* algorithmic_flops, double* kind_ms) {
  double ms = 0, fl = 0, km[3] = {0, 0, 0};
  for (int i = 0; i < g_ntimed; ++i) {
    NB_CUDA(cudaEventSynchronize(g_timed[i].b));
    float t = 0;
    NB_CUDA(cudaEventElapsedTime(&t, g_timed[i].a, g_timed[i].b));
    ms += t; fl += g_timed[i].flops;
    if (g_timed[i].kind >= 0 && g_timed[i].kind < 3) km[g_timed[i].kind] += t;
    cudaEventDestroy(g_timed[i].a); cudaEventDestroy(g_timed[i].b);
  }
  if (kernel_ms) *kernel_ms = ms;
  if (launches) *launches = g_ntimed;
  if (algorithmic_flops) *algorithmic_flops = fl;
  if (kind_ms) { kind_ms[0] = km[0]; kind_ms[1] = km[1]; kind_ms[2] = km[2]; }
  g_ntimed = 0;
  return 0;
}

int nerf_b200_embed(const float* x, int64_t M, int L, float* out, void* stream) {
  NB_CHECK_ARG(x && out, "NULL pointer");
  NB_CHECK_ARG(L >= 0 && L <= 16, "num_freqs out of range");
  if (M == 0) return 0;
  long long total = M * (3 + 6 * L);
  embed_kernel<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(x, M, L, out);
  NB_LAUNCH_OK("embed_kernel");
  return 0;
}

size_t nerf_b200_packed_bytes(const NerfNetParams* net) {
  if (!net || check_tc_net(net)) return 0;
  return make_pack_layout(*net).total;
}

int nerf_b200_pack_weights(const NerfNetParams* net, void* packed, size_t packed_bytes, void* stream) {
  if (int rc = check_tc_net(net)) return rc;
  const PackLayout PL = make_pack_layout(*net);
  NB_CHECK_ARG(packed && packed_bytes >= PL.total, "packed buffer too small (%zu < %zu)", packed_bytes, PL.total);
  cudaStream_t st = (cudaStream_t)stream;
  PackJob job;
  job.n = 0;
  unsigned off = (unsigned)PL.off_chunks;
  const int IC = net->input_ch, W = net->W;
  auto add = [&](const float* src, int ld, int k0, int kvalid, int nrows) {
    PackChunk& c = job.c[job.n++];
    c.src = src; c.sn = ld; c.sk = 1; c.k0 = k0; c.kvalid = kvalid < 0 ? 0 : (kvalid > 32 ? 32 : kvalid); c.nrows = nrows; c.dst_off = off;
    off += (unsigned)nrows * 64;
  };
  PackBiasJob bj;
  bj.n = 0;
  for (int l = 0; l < PL.NL; ++l) {
    if (tc_layer_has_bias(l, net->D)) bj.src[bj.n++] = (l < net->D) ? net->pts_b[l] : net->feature_b;
    if (l == 0) { add(net->pts_w[0], IC, 0, IC, 256); add(net->pts_w[0], IC, 32, IC - 32, 256); }
    else if (l < net->D) {
      const bool sk = (net->skip >= 0 && l == net->skip + 1);
      const int ld = sk ? W + IC : W, base = sk ? IC : 0;
      if (sk) { add(net->pts_w[l], ld, 0, IC, 256); add(net->pts_w[l], ld, 32, IC - 32, 256); }    // cat([input_pts, h])
      for (int c = 0; c < 8; ++c) add(net->pts_w[l], ld, base + 32 * c, 32, 256);
    } else if (l == net->D) { for (int c = 0; c < 8; ++c) add(net->feature_w, W, 32 * c, 32, 256); }
    else { for (int c = 0; c < 8; ++c) add(net->views_w, W + net->input_ch_views, 32 * c, 32, 128); }
  }
  NB_CHECK_ARG(job.n == PL.n_chunks && off == PL.off_chunks + PL.chunk_bytes, "internal: chunk table mismatch");
  bj.dst_off = (unsigned)PL.off_biasb;
  pack_bias_kernel<<<1, 256, 0, st>>>(bj, static_cast<uint8_t*>(packed));
  NB_LAUNCH_OK("pack_bias_kernel");
  dim3 grid(4, job.n);
  pack_chunks_kernel<<<grid, 256, 0, st>>>(job, static_cast<uint8_t*>(packed));
  NB_LAUNCH_OK("pack_chunks_kernel");
  {
    // rank-split copy for the CTA-pair kernel: [rank 0: every chunk's rows 0..N/2-1][rank 1: rows N/2..N-1], so that
    // two consecutive chunk halves of one CTA are contiguous (one 16 KB TMA box)
    uint8_t* base = static_cast<uint8_t*>(packed);
    const size_t views_bytes = net->use_viewdirs ? (size_t)8 * (TC_STAGE_BYTES / 2) : 0;
    const size_t reg_bytes = PL.chunk_bytes - views_bytes;
    for (int r = 0; r < 2; ++r) {
      uint8_t* dst = base + PL.off_pair + (size_t)r * (PL.chunk_bytes / 2);
      NB_CUDA(cudaMemcpy2DAsync(dst, 8192, base + PL.off_chunks + (size_t)r * 8192, 16384, 8192, reg_bytes / 16384, cudaMemcpyDeviceToDevice, st));
      if (views_bytes)
        NB_CUDA(cudaMemcpy2DAsync(dst + reg_bytes / 2, 4096, base + PL.off_chunks + reg_bytes + (size_t)r * 4096, 8192, 4096, 8, cudaMemcpyDeviceToDevice, st));
    }
  }
  if (PL.bwd_bytes) {
    // backward (dgrad) stream, bwd_tc2.cuh: chunk [n][k] = W[k0 + k][col0 + n] -- the transposed weights, so that the
    // chain dA_{l-1} = dA_l W_l runs through the forward's operand layouts.  Step 0: views_linears[0].weight[:, :W]
    // (K = W/2), step 1: feature_linear, then pts_linears[D-1] ... [1] restricted to their h columns.
    PackJob bj2;
    bj2.n = 0;
    unsigned boff = (unsigned)PL.off_bwd;
    auto addT = [&](const float* src, int ld, int col0, int k0) {
      PackChunk& c = bj2.c[bj2.n++];
      c.src = src + col0; c.sn = 1; c.sk = ld; c.k0 = k0; c.kvalid = 32; c.nrows = 256; c.dst_off = boff;
      boff += 256u * 64u;
    };
    for (int c = 0; c < 4; ++c) addT(net->views_w, W + net->input_ch_views, 0, 32 * c);
    for (int c = 0; c < 8; ++c) addT(net->feature_w, W, 0, 32 * c);
    for (int l = net->D - 1; l >= 1; --l) {
      const bool sk = (net->skip >= 0 && l == net->skip + 1);
      for (int c = 0; c < 8; ++c) addT(net->pts_w[l], sk ? W + IC : W, sk ? IC : 0, 32 * c);
    }
    NB_CHECK_ARG(bj2.n == 4 + 8 * net->D && boff == PL.off_bwd + PL.bwd_bytes, "internal: backward chunk table mismatch");
    dim3 g2(4, bj2.n);
    pack_chunks_kernel<<<g2, 256, 0, st>>>(bj2, static_cast<uint8_t*>(packed));
    NB_LAUNCH_OK("pack_chunks_kernel (backward stream)");
    uint8_t* base = static_cast<uint8_t*>(packed);
    for (int r = 0; r < 2; ++r)
      NB_CUDA(cudaMemcpy2DAsync(base + PL.off_bwd_pair + (size_t)r * (PL.bwd_bytes / 2), 8192, base + PL.off_bwd + (size_t)r * 8192, 16384, 8192,
                                PL.bwd_bytes / 16384, cudaMemcpyDeviceToDevice, st));
  }
  PackTables t;
  t.net = *net; t.off_bias = PL.off_bias; t.off_heads = PL.off_heads; t.off_vdir = PL.off_vdir;
  pack_tables_kernel<<<8, 256, 0, st>>>(t, static_cast<uint8_t*>(packed));
  NB_LAUNCH_OK("pack_tables_kernel");
  return 0;
}

int nerf_b200_run_network(const float* pts, const float* viewdirs, int64_t N, int S, const NerfNetParams* net,
                          const void* packed, int multires, int multires_views, int precision, float* raw,
                          void* workspace, size_t workspace_bytes, void* stream) {
  NB_CHECK_ARG(pts && raw && net, "NULL pointer");
  if (N == 0 || S == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  if (precision == NERF_B200_PREC_FP32) {
    NB_CHECK_ARG(net->W <= SIMT_THREADS && net->W % 4 == 0, "exact path supports netwidth <= 256");
    NB_CHECK_ARG(!net->use_viewdirs || viewdirs, "viewdirs required");
    const long long M = N * (long long)S;
    const size_t sm = simt_smem_bytes(*net);
    if (int rc = smem_optin((const void*)mlp_simt_kernel, sm)) return rc;
    mlp_simt_kernel<<<cdiv(M, SIMT_ROWS), SIMT_THREADS, sm, st>>>(pts, viewdirs, 3, M, S, *net, multires, multires_views, raw, SimtSave{});
    NB_LAUNCH_OK("mlp_simt_kernel");
    return 0;
  }
  NB_CHECK_ARG(precision == NERF_B200_PREC_TC_FP16, "unknown precision %d", precision);
  NerfPassOut out;
  memset(&out, 0, sizeof(out));
  out.raw = raw;
  return launch_march(nullptr, 0, nullptr, pts, viewdirs, 3, nullptr, N, S, net, packed, multires, multires_views, 0, 0,
                      &out, workspace, workspace_bytes, nullptr, nullptr, st);
}

int nerf_b200_raw2outputs(const float* raw, const float* z_vals, const float* rays_d, int d_stride, const float* noise,
                          int64_t N, int S, int white_bkgd, const NerfPassOut* out, void* stream) {
  NB_CHECK_ARG(raw && z_vals && rays_d && out, "NULL pointer");
  NB_CHECK_ARG(S >= 1, "S must be >= 1");
  if (N == 0) return 0;
  raw2outputs_kernel<<<cdiv(N * 32, 256), 256, 0, (cudaStream_t)stream>>>(raw, z_vals, rays_d, d_stride, noise, N, S, white_bkgd, *out);
  NB_LAUNCH_OK("raw2outputs_kernel");
  return 0;
}

int nerf_b200_raw2outputs_bwd(const float* raw, const float* z_vals, const float* rays_d, int d_stride, const float* noise,
                              int64_t N, int S, int white_bkgd, const float* g_rgb, float* d_raw, void* stream) {
  NB_CHECK_ARG(raw && z_vals && rays_d && g_rgb && d_raw, "NULL pointer");
  NB_CHECK_ARG(S >= 1 && S <= 1024, "S must be in [1,1024]");
  if (N == 0) return 0;
  const int wpb = 4;
  const size_t sm = (size_t)wpb * 4 * S * sizeof(float);
  if (int rc = smem_optin((const void*)raw2outputs_bwd_kernel, sm)) return rc;
  raw2outputs_bwd_kernel<<<cdiv(N, wpb), wpb * 32, sm, (cudaStream_t)stream>>>(raw, z_vals, rays_d, d_stride, noise, N, S, white_bkgd, g_rgb, d_raw);
  NB_LAUNCH_OK("raw2outputs_bwd_kernel");
  return 0;
}

static int fill_pack_args(PackRaysArgs& a, const float* rays_o, const float* rays_d, const float* view_src, const NerfCamera* cam, int64_t N,
                          int64_t pixel0, const int64_t* pixel_index, int ndc, float near, float far, int use_viewdirs) {
  NB_CHECK_ARG((rays_o && rays_d) || (cam && !rays_o && !rays_d), "give rays_o and rays_d, or a camera to generate them");
  NB_CHECK_ARG(!ndc || cam, "ndc needs the camera (H, W, focal)");
  memset(&a, 0, sizeof(a));
  a.rays_o = rays_o; a.rays_d = rays_d; a.view_src = view_src; a.N = N; a.pixel0 = pixel0;
  a.pixel_index = reinterpret_cast<const long long*>(pixel_index);
  a.ndc = ndc; a.use_viewdirs = use_viewdirs; a.stride = use_viewdirs ? 11 : 8; a.near = near; a.far = far;
  if (cam) {
    a.H = cam->H; a.W = cam->W; a.fx = cam->fx; a.fy = cam->fy; a.cx = cam->cx; a.cy = cam->cy;
    memcpy(a.c2w, cam->c2w, sizeof(a.c2w));
    a.ndc_cw = (float)(-1.0 / ((double)cam->W / (2.0 * (double)cam->fx)));      // run_nerf_helpers.py:181 (focal = K[0][0])
    a.ndc_ch = (float)(-1.0 / ((double)cam->H / (2.0 * (double)cam->fx)));
  }
  return 0;
}

static int pack_rays_impl(const float* rays_o, const float* rays_d, const float* view_src, const NerfCamera* cam, int64_t N,
                          int64_t pixel0, const int64_t* pixel_index, int ndc, float near, float far, int use_viewdirs, float* out, void* stream) {
  NB_CHECK_ARG(out != nullptr, "NULL output");
  if (N == 0) return 0;
  PackRaysArgs a;
  if (int rc = fill_pack_args(a, rays_o, rays_d, view_src, cam, N, pixel0, pixel_index, ndc, near, far, use_viewdirs)) return rc;
  pack_rays_kernel<<<cdiv(N, 256), 256, 0, (cudaStream_t)stream>>>(a, out);
  NB_LAUNCH_OK("pack_rays_kernel");
  return 0;
}

int nerf_b200_pack_rays(const float* rays_o, const float* rays_d, const float* view_src, const NerfCamera* cam, int64_t N,
                        int64_t pixel0, int ndc, float near, float far, int use_viewdirs, float* out, void* stream) {
  return pack_rays_impl(rays_o, rays_d, view_src, cam, N, pixel0, nullptr, ndc, near, far, use_viewdirs, out, stream);
}

// the same for an arbitrary list of pixels of the camera's image (the per-image random pixel choice of run_nerf.py:728-757,
// without materialising get_rays' [H, W, 3] tensors or gathering from them)
int nerf_b200_pack_rays_pixels(const NerfCamera* cam, const int64_t* pixel_index, int64_t N, int ndc, float near, float far,
                               int use_viewdirs, float* out, void* stream) {
  NB_CHECK_ARG(cam && pixel_index, "camera and pixel_index are required");
  return pack_rays_impl(nullptr, nullptr, nullptr, cam, N, 0, pixel_index, ndc, near, far, use_viewdirs, out, stream);
}

int nerf_b200_to8b(const float* x, int64_t n, uint8_t* out, void* stream) {
  NB_CHECK_ARG(x && out, "NULL pointer");
  if (n == 0) return 0;
  to8b_kernel<<<cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>(x, n, out);
  NB_LAUNCH_OK("to8b_kernel");
  return 0;
}

int nerf_b200_sample_pdf(const float* bins, const float* weights, const float* u, int64_t u_row_stride, int64_t N, int B,
                         int n_samples, float* samples, void* stream) {
  NB_CHECK_ARG(bins && weights && u && samples, "NULL pointer");
  NB_CHECK_ARG(B >= 2 && B <= 2048 && n_samples >= 1, "bad B / n_samples");
  if (N == 0) return 0;
  const int wpb = 4;
  const size_t sm = (size_t)wpb * 3 * B * sizeof(float);
  if (int rc = smem_optin((const void*)sample_pdf_kernel, sm)) return rc;
  sample_pdf_kernel<<<cdiv(N, wpb), wpb * 32, sm, (cudaStream_t)stream>>>(bins, weights, u, u_row_stride, N, B, n_samples, samples);
  NB_LAUNCH_OK("sample_pdf_kernel");
  return 0;
}

int nerf_b200_coarse_z(const float* rays, int ray_stride, const float* t_vals, const float* t_rand, int64_t N, int S,
                       int lindisp, float* z_vals, void* stream) {
  NB_CHECK_ARG(rays && t_vals && z_vals, "NULL pointer");
  NB_CHECK_ARG(ray_stride >= 8, "ray_stride must be >= 8");
  if (N == 0) return 0;
  coarse_z_kernel<<<cdiv(N * S, 256), 256, 0, (cudaStream_t)stream>>>(rays, ray_stride, t_vals, t_rand, N, S, lindisp, z_vals);
  NB_LAUNCH_OK("coarse_z_kernel");
  return 0;
}

int nerf_b200_fine_z(const float* z_vals, const float* weights, const float* u, int64_t u_row_stride, int64_t N, int S,
                     int n_imp, float* z_fine, float* z_samples, float* z_std, void* stream) {
  NB_CHECK_ARG(z_vals && weights && u && z_fine, "NULL pointer");
  NB_CHECK_ARG(S >= 3 && n_imp >= 1 && S + n_imp <= 4096, "bad S / n_imp");
  if (N == 0) return 0;
  int P = 1;
  while (P < S + n_imp) P <<= 1;
  const int wpb = 4;
  const size_t sm = (size_t)wpb * (3 * S + P) * sizeof(float);
  if (int rc = smem_optin((const void*)fine_z_kernel, sm)) return rc;
  fine_z_kernel<<<cdiv(N, wpb), wpb * 32, sm, (cudaStream_t)stream>>>(z_vals, weights, u, u_row_stride, N, S, n_imp, P, z_fine, z_samples, z_std);
  NB_LAUNCH_OK("fine_z_kernel");
  return 0;
}

size_t nerf_b200_march_workspace_bytes(int64_t N, int S) {
  size_t tc = (size_t)N * 128 * 4 * 2, exact = (size_t)N * S * 28;   // view-bias tables of both nets | pts + raw scratch
  return (tc > exact ? tc : exact) + 256;
}

static int march_impl(const float* rays, const float* z_vals, const float* noise, int64_t N, int S, const NerfNetParams* net,
                      const void* packed, const NerfRenderCfg* cfg, const NerfPassOut* out, void* workspace,
                      size_t workspace_bytes, const NerfTrainSave* save, void* stream, const float* vb_pre = nullptr) {
  NB_CHECK_ARG(rays && z_vals && net && cfg && out, "NULL pointer");
  if (N == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  NB_CHECK_ARG(cfg->ray_stride >= (net->use_viewdirs ? 11 : 8), "ray_stride %d too small", cfg->ray_stride);
  if (cfg->precision == NERF_B200_PREC_FP32) {
    // exact mode (validation path): materialise pts -> fp32 CUDA-core MLP -> raw2outputs kernel
    NB_CHECK_ARG(save == nullptr, "training-mode records belong to the tensor-core path");
    const long long M = N * (long long)S;
    const size_t need = (size_t)M * 12 + (out->raw ? 0 : (size_t)M * 16);
    NB_CHECK_ARG(workspace && workspace_bytes >= need, "exact-mode workspace too small: need %zu bytes", need);
    NB_CHECK_ARG(net->W <= SIMT_THREADS && net->W % 4 == 0, "exact path supports netwidth <= 256");
    float* pts = static_cast<float*>(workspace);
    float* raw = out->raw ? out->raw : pts + (size_t)M * 3;
    pts_kernel<<<cdiv(M, 256), 256, 0, st>>>(rays, cfg->ray_stride, z_vals, M, S, pts);
    NB_LAUNCH_OK("pts_kernel");
    const size_t sm = simt_smem_bytes(*net);
    if (int rc = smem_optin((const void*)mlp_simt_kernel, sm)) return rc;
    mlp_simt_kernel<<<cdiv(M, SIMT_ROWS), SIMT_THREADS, sm, st>>>(pts, rays + 8, cfg->ray_stride, M, S, *net, cfg->multires, cfg->multires_views, raw, SimtSave{});
    NB_LAUNCH_OK("mlp_simt_kernel");
    raw2outputs_kernel<<<cdiv(N * 32, 256), 256, 0, st>>>(raw, z_vals, rays + 3, cfg->ray_stride, noise, N, S, cfg->white_bkgd, *out);
    NB_LAUNCH_OK("raw2outputs_kernel");
    return 0;
  }
  return launch_march(rays, cfg->ray_stride, z_vals, nullptr, rays + 8, cfg->ray_stride, noise, N, S, net, packed,
                      cfg->multires, cfg->multires_views, cfg->white_bkgd, 1, out, workspace, workspace_bytes, save, vb_pre, st);
}

int nerf_b200_march(const float* rays, const float* z_vals, const float* noise, int64_t N, int S, const NerfNetParams* net,
                    const void* packed, const NerfRenderCfg* cfg, const NerfPassOut* out, void* workspace,
                    size_t workspace_bytes, void* stream) {
  return march_impl(rays, z_vals, noise, N, S, net, packed, cfg, out, workspace, workspace_bytes, nullptr, stream);
}

int nerf_b200_march_train(const float* rays, const float* z_vals, const float* noise, int64_t N, int S, const NerfNetParams* net,
                          const void* packed, const NerfRenderCfg* cfg, const NerfPassOut* out, void* workspace,
                          size_t workspace_bytes, const NerfTrainSave* save, void* stream) {
  NB_CHECK_ARG(save != nullptr && out && out->raw, "training mode needs the save buffers and out->raw (the compositing adjoint reads raw)");
  return march_impl(rays, z_vals, noise, N, S, net, packed, cfg, out, workspace, workspace_bytes, save, stream);
}

int nerf_b200_train_record_bytes(int64_t N, int S, const NerfNetParams* net, size_t* act_bytes, size_t* mask_bytes) {
  if (int rc = check_tc_net(net)) return rc;
  NB_CHECK_ARG(N >= 0 && S >= 1, "bad N / S");
  const TilePlan plan = make_tile_plan(N > 0 ? N : 1, S, num_sms());
  if (act_bytes) *act_bytes = (size_t)plan.n_tiles * rec_act_bytes(net->D);
  if (mask_bytes) *mask_bytes = (size_t)plan.n_tiles * rec_mask_bytes(net->D);
  return 0;
}

static int render_rays_fwd_impl(const float* rays, int64_t N, const NerfRenderCfg* cfg, const NerfNetParams* net_coarse,
                                const void* packed_coarse, const NerfNetParams* net_fine, const void* packed_fine,
                                const float* t_vals, const float* u_det, const float* t_rand, const float* u_rand,
                                const float* noise0, const float* noise1, float* z_coarse, const NerfPassOut* coarse,
                                float* z_fine, float* z_std, const NerfPassOut* fine, void* workspace,
                                size_t workspace_bytes, const NerfTrainSave* save_coarse, const NerfTrainSave* save_fine, void* stream,
                                const NerfRayGen* gen = nullptr) {
  NB_CHECK_ARG(rays && cfg && net_coarse && t_vals && z_coarse && coarse, "NULL pointer");
  if (N == 0) return 0;
  // gen: `rays` is still to be built (render()'s batch construction, run_nerf.py:95-123) -- by the prologue kernel below on the
  // tensor-core path, by pack_rays_kernel otherwise
  PackRaysArgs pk;
  bool pack_pending = false;
  if (gen) {
    NB_CHECK_ARG(cfg->ray_stride == (gen->use_viewdirs ? 11 : 8), "ray_stride does not match the batch to build");
    if (int rc = fill_pack_args(pk, gen->rays_o, gen->rays_d, gen->view_src, gen->cam, N, gen->pixel0, nullptr, gen->ndc, gen->near, gen->far, gen->use_viewdirs)) return rc;
    pack_pending = true;
  }
  const int Sc = cfg->N_samples, Ni = cfg->N_importance;
  NB_CHECK_ARG(Sc >= 1 && Ni >= 0, "bad sample counts");
  NB_CHECK_ARG(!cfg->perturb || t_rand, "perturb > 0 needs t_rand");
  // per-ray prologue: z sampling (run_nerf.py:357-379) and, on the tensor-core path, the view-bias tables of both networks
  // -- one launch (ray_setup_kernel); the exact path keeps the stand-alone z kernel
  const NerfNetParams* nf = net_fine ? net_fine : net_coarse;
  const void* pf = net_fine ? packed_fine : packed_coarse;
  const float* vb_c = nullptr;
  const float* vb_f = nullptr;
  if (cfg->precision == NERF_B200_PREC_TC_FP16 && net_coarse->use_viewdirs && packed_coarse && (Ni == 0 || (nf->use_viewdirs && pf))) {
    if (int rc = check_tc_net(net_coarse)) return rc;
    NB_CHECK_ARG(workspace != nullptr && workspace_bytes >= (size_t)N * 128 * 4 * 2, "workspace too small: need %zu bytes", (size_t)N * 128 * 4 * 2);
    NB_CHECK_ARG(cfg->ray_stride >= 11, "ray_stride %d too small for view directions", cfg->ray_stride);
    NB_CHECK_ARG(3 + 6 * cfg->multires_views == net_coarse->input_ch_views || (cfg->multires_views == 0 && net_coarse->input_ch_views == 3), "multires_views mismatch");
    const PackLayout PLc = make_pack_layout(*net_coarse);
    RaySetupArgs a;
    memset(&a, 0, sizeof(a));
    a.rays = rays; a.ray_stride = cfg->ray_stride; a.N = N; a.Lv = cfg->multires_views; a.ICV = net_coarse->input_ch_views;
    float* vb = static_cast<float*>(workspace);
    a.vdir_a = reinterpret_cast<const float*>(static_cast<const uint8_t*>(packed_coarse) + PLc.off_vdir); a.vb_a = vb;
    vb_c = vb;
    if (Ni > 0) {
      if (nf == net_coarse || pf == packed_coarse) vb_f = vb_c;
      else {
        NB_CHECK_ARG(nf->input_ch_views == net_coarse->input_ch_views, "coarse and fine networks must encode view directions alike");
        const PackLayout PLf = make_pack_layout(*nf);
        a.vdir_b = reinterpret_cast<const float*>(static_cast<const uint8_t*>(pf) + PLf.off_vdir); a.vb_b = vb + (size_t)N * 128;
        vb_f = a.vb_b;
      }
    }
    a.t_vals = t_vals; a.t_rand = cfg->perturb ? t_rand : nullptr; a.S = Sc; a.lindisp = cfg->lindisp; a.z_out = z_coarse;
    if (pack_pending) { a.pack = pk; a.pack_out = const_cast<float*>(rays); pack_pending = false; }
    ray_setup_kernel<<<cdiv(N, VB_RAYS), 256, 0, (cudaStream_t)stream>>>(a);
    NB_LAUNCH_OK("ray_setup_kernel");
  } else {
    if (pack_pending) {
      pack_rays_kernel<<<cdiv(N, 256), 256, 0, (cudaStream_t)stream>>>(pk, const_cast<float*>(rays));
      NB_LAUNCH_OK("pack_rays_kernel");
    }
    if (int rc = nerf_b200_coarse_z(rays, cfg->ray_stride, t_vals, cfg->perturb ? t_rand : nullptr, N, Sc, cfg->lindisp, z_coarse, stream)) return rc;
  }
  // coarse pass (:381-386)
  if (int rc = march_impl(rays, z_coarse, noise0, N, Sc, net_coarse, packed_coarse, cfg, coarse, workspace, workspace_bytes, save_coarse, stream, vb_c)) return rc;
  if (Ni == 0) return 0;
  NB_CHECK_ARG(coarse->weights && z_fine && fine, "N_importance > 0 needs coarse->weights, z_fine and fine outputs");
  // hierarchical sampling (:392-396, :412); det <=> perturb == 0 (:393)
  const float* u = cfg->perturb ? u_rand : u_det;
  NB_CHECK_ARG(u != nullptr, "missing u (u_det for perturb==0, u_rand otherwise)");
  if (int rc = nerf_b200_fine_z(z_coarse, coarse->weights, u, cfg->perturb ? Ni : 0, N, Sc, Ni, z_fine, nullptr, z_std, stream)) return rc;
  // fine pass on all S_c + N_importance samples (:397-403); network_fine None -> coarse net (:399)
  return march_impl(rays, z_fine, noise1, N, Sc + Ni, nf, pf, cfg, fine, workspace, workspace_bytes, save_fine, stream, vb_f);
}

int nerf_b200_render_rays_fwd(const float* rays, int64_t N, const NerfRenderCfg* cfg, const NerfNetParams* net_coarse,
                              const void* packed_coarse, const NerfNetParams* net_fine, const void* packed_fine,
                              const float* t_vals, const float* u_det, const float* t_rand, const float* u_rand,
                              const float* noise0, const float* noise1, float* z_coarse, const NerfPassOut* coarse,
                              float* z_fine, float* z_std, const NerfPassOut* fine, void* workspace,
                              size_t workspace_bytes, void* stream) {
  return render_rays_fwd_impl(rays, N, cfg, net_coarse, packed_coarse, net_fine, packed_fine, t_vals, u_det, t_rand, u_rand, noise0, noise1,
                              z_coarse, coarse, z_fine, z_std, fine, workspace, workspace_bytes, nullptr, nullptr, stream);
}

// render() for one chunk: the ray batch is BUILT (get_rays / viewdirs / NDC / near-far / packing, run_nerf.py:95-123) by the same
// prologue launch that samples z and fills the view-bias tables, into `rays` [N, 8 | 11], then rendered as above
int nerf_b200_render_fwd(const NerfRayGen* gen, float* rays, int64_t N, const NerfRenderCfg* cfg, const NerfNetParams* net_coarse,
                         const void* packed_coarse, const NerfNetParams* net_fine, const void* packed_fine,
                         const float* t_vals, const float* u_det, const float* t_rand, const float* u_rand,
                         const float* noise0, const float* noise1, float* z_coarse, const NerfPassOut* coarse,
                         float* z_fine, float* z_std, const NerfPassOut* fine, void* workspace,
                         size_t workspace_bytes, void* stream) {
  NB_CHECK_ARG(gen != nullptr, "NULL ray generator");
  return render_rays_fwd_impl(rays, N, cfg, net_coarse, packed_coarse, net_fine, packed_fine, t_vals, u_det, t_rand, u_rand, noise0, noise1,
                              z_coarse, coarse, z_fine, z_std, fine, workspace, workspace_bytes, nullptr, nullptr, stream, gen);
}

// the same call in training mode: both passes also leave their per-tile records (activation images + ReLU masks) for
// nerf_b200_march_bwd_tc, and must write raw (coarse->raw, fine->raw)
int nerf_b200_render_rays_fwd_train(const float* rays, int64_t N, const NerfRenderCfg* cfg, const NerfNetParams* net_coarse,
                                    const void* packed_coarse, const NerfNetParams* net_fine, const void* packed_fine,
                                    const float* t_vals, const float* u_det, const float* t_rand, const float* u_rand,
                                    const float* noise0, const float* noise1, float* z_coarse, const NerfPassOut* coarse,
                                    float* z_fine, float* z_std, const NerfPassOut* fine, void* workspace,
                                    size_t workspace_bytes, const NerfTrainSave* save_coarse, const NerfTrainSave* save_fine, void* stream) {
  NB_CHECK_ARG(cfg && cfg->precision == NERF_B200_PREC_TC_FP16, "training-mode records belong to the tensor-core path");
  NB_CHECK_ARG(save_coarse && coarse && coarse->raw, "training mode needs save_coarse and coarse->raw");
  NB_CHECK_ARG(cfg->N_importance == 0 || (save_fine && fine && fine->raw), "training mode needs save_fine and fine->raw");
  return render_rays_fwd_impl(rays, N, cfg, net_coarse, packed_coarse, net_fine, packed_fine, t_vals, u_det, t_rand, u_rand, noise0, noise1,
                              z_coarse, coarse, z_fine, z_std, fine, workspace, workspace_bytes, save_coarse, save_fine, stream);
}

// ---- exact-mode backward of one pass (see bwd_simt.cuh) -------------------------------------------
static const int BWD_RAYS_PER_SLAB = 512;     // rays recomputed + back-propagated per slab (bounds the workspace)

size_t nerf_b200_march_bwd_workspace_bytes(int64_t N, int S, const NerfNetParams* net) {
  if (!net) return 0;
  const long long rows = (long long)(N < BWD_RAYS_PER_SLAB ? N : BWD_RAYS_PER_SLAB) * S;
  return (size_t)rows * (3 + bwd_floats_per_row(*net)) * 4 + 1024;
}

static int gemm_nn(const float* A, int lda, const float* B, int ldb, float* C, int ldc, long long M, int N, int K, int beta, cudaStream_t st) {
  dim3 grid(cdiv(M, GT), cdiv(N, GT));
  sgemm_nn_kernel<<<grid, 256, 0, st>>>(A, lda, B, ldb, C, ldc, M, N, K, beta);
  NB_LAUNCH_OK("sgemm_nn_kernel");
  return 0;
}
static int gemm_tn(const float* A, int lda, const float* B, int ldb, float* C, int ldc, long long M, int K1, int N, cudaStream_t st) {
  const int slab = 2048;
  dim3 grid(cdiv(K1, GT), cdiv(N, GT), cdiv(M, slab));
  sgemm_tn_kernel<<<grid, 256, 0, st>>>(A, lda, B, ldb, C, ldc, M, K1, N, slab);
  NB_LAUNCH_OK("sgemm_tn_kernel");
  return 0;
}
static int mask_colsum(float* d, int ldd, const float* h, int ldh, long long M, int C, float* colsum, cudaStream_t st) {
  const int rpb = 256;
  dim3 grid(cdiv(M, rpb), cdiv(C, 64));
  relu_mask_colsum_kernel<<<grid, 64, 0, st>>>(d, ldd, h, ldh, M, C, colsum, rpb);
  NB_LAUNCH_OK("relu_mask_colsum_kernel");
  return 0;
}
#define NB_TRY(expr) do { if (int rc__ = (expr)) return rc__; } while (0)

int nerf_b200_march_bwd(const float* rays, const float* z_vals, const float* noise, int64_t N, int S, const NerfNetParams* net,
                        const void* packed, const NerfRenderCfg* cfg, const float* g_rgb, const NerfNetGrads* grads,
                        void* workspace, size_t workspace_bytes, void* stream) {
  (void)packed;
  NB_CHECK_ARG(rays && z_vals && net && cfg && g_rgb && grads, "NULL pointer");
  NB_CHECK_ARG(net->W <= SIMT_THREADS && net->W % 4 == 0 && net->D <= NERF_B200_MAX_D, "unsupported network shape");
  if (N == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  const int W = net->W, W2 = W / 2, IC = net->input_ch, ICV = net->input_ch_views, D = net->D, rs = cfg->ray_stride;
  NB_CHECK_ARG(workspace && workspace_bytes >= nerf_b200_march_bwd_workspace_bytes(N, S, net), "march_bwd workspace too small");
  for (int64_t n0 = 0; n0 < N; n0 += BWD_RAYS_PER_SLAB) {
    const int64_t nn = (N - n0 < BWD_RAYS_PER_SLAB) ? N - n0 : BWD_RAYS_PER_SLAB;
    const long long M = nn * (long long)S;
    const float* ry = rays + n0 * rs;
    const float* zz = z_vals + n0 * S;
    const float* nz = noise ? noise + n0 * S : nullptr;
    float* p = static_cast<float*>(workspace);
    float* pts = p;        p += M * 3;
    SimtSave sv;
    sv.enc = p;            p += M * IC;
    sv.encv = p;           p += M * ICV;
    sv.h = p;              p += (size_t)D * M * W;
    sv.feat = p;           p += M * W;
    sv.hv = p;             p += M * W2;
    float* raw = p;        p += M * 4;
    float* d_raw = p;      p += M * 4;
    float* dh0 = p;        p += M * W;
    float* dh1 = p;        p += M * W;
    float* d_hv = p;       p += M * W2;
    if (!net->use_viewdirs) { sv.encv = nullptr; sv.feat = nullptr; sv.hv = nullptr; }
    // 1. recompute the pass in fp32 with saved activations
    pts_kernel<<<cdiv(M, 256), 256, 0, st>>>(ry, rs, zz, M, S, pts);
    NB_LAUNCH_OK("pts_kernel");
    const size_t sm = simt_smem_bytes(*net);
    NB_TRY(smem_optin((const void*)mlp_simt_kernel, sm));
    mlp_simt_kernel<<<cdiv(M, SIMT_ROWS), SIMT_THREADS, sm, st>>>(pts, net->use_viewdirs ? ry + 8 : nullptr, rs, M, S, *net, cfg->multires, cfg->multires_views, raw, sv);
    NB_LAUNCH_OK("mlp_simt_kernel");
    // 2. compositing adjoint -> dL/draw
    NB_TRY(nerf_b200_raw2outputs_bwd(raw, zz, ry + 3, rs, nz, nn, S, cfg->white_bkgd, g_rgb + n0 * 3, d_raw, stream));
    const float* h_last = sv.h + (size_t)(D - 1) * M * W;
    if (net->use_viewdirs) {
      // 3. rgb_linear (run_nerf_helpers.py:114)
      NB_TRY(gemm_tn(d_raw, 4, sv.hv, W2, grads->rgb_w, W2, M, 3, W2, st));
      NB_TRY(mask_colsum(d_raw, 4, nullptr, 0, M, 3, grads->rgb_b, st));
      NB_TRY(gemm_nn(d_raw, 4, net->rgb_w, W2, d_hv, W2, M, W2, 3, 0, st));
      // 4. views_linears[0] on cat([feature, input_views]) (:108-112)
      NB_TRY(mask_colsum(d_hv, W2, sv.hv, W2, M, W2, grads->views_b, st));
      NB_TRY(gemm_tn(d_hv, W2, sv.feat, W, grads->views_w, W + ICV, M, W2, W, st));
      NB_TRY(gemm_tn(d_hv, W2, sv.encv, ICV, grads->views_w + W, W + ICV, M, W2, ICV, st));
      NB_TRY(gemm_nn(d_hv, W2, net->views_w, W + ICV, dh0, W, M, W, W2, 0, st));                // d_feature
      // 5. feature_linear and alpha_linear both read the last hidden layer (:106-107)
      NB_TRY(gemm_tn(dh0, W, h_last, W, grads->feature_w, W, M, W, W, st));
      NB_TRY(mask_colsum(dh0, W, nullptr, 0, M, W, grads->feature_b, st));
      NB_TRY(gemm_tn(d_raw + 3, 4, h_last, W, grads->alpha_w, W, M, 1, W, st));
      NB_TRY(mask_colsum(d_raw + 3, 4, nullptr, 0, M, 1, grads->alpha_b, st));
      NB_TRY(gemm_nn(dh0, W, net->feature_w, W, dh1, W, M, W, W, 0, st));
      NB_TRY(gemm_nn(d_raw + 3, 4, net->alpha_w, W, dh1, W, M, W, 1, 1, st));
    } else {
      // 3'. output_linear (:117): only its first four rows ever reach the loss (run_nerf.py:187 note); rows >= 4 get zero gradient
      NB_TRY(gemm_tn(d_raw, 4, h_last, W, grads->output_w, W, M, 4, W, st));
      NB_TRY(mask_colsum(d_raw, 4, nullptr, 0, M, 4, grads->output_b, st));
      NB_TRY(gemm_nn(d_raw, 4, net->output_w, W, dh1, W, M, W, 4, 0, st));
    }
    // 6. pts_linears, last to first (:99-103); skip layer input = cat([input_pts, h])
    float* dcur = dh1;
    float* dnext = dh0;
    for (int l = D - 1; l >= 0; --l) {
      NB_TRY(mask_colsum(dcur, W, sv.h + (size_t)l * M * W, W, M, W, grads->pts_b[l], st));
      const bool after_skip = (l > 0) && (l - 1 == net->skip);
      const int Kl = (l == 0) ? IC : (after_skip ? W + IC : W);
      if (l == 0) {
        NB_TRY(gemm_tn(dcur, W, sv.enc, IC, grads->pts_w[0], Kl, M, W, IC, st));
      } else {
        const float* hprev = sv.h + (size_t)(l - 1) * M * W;
        const int off = after_skip ? IC : 0;
        if (after_skip) NB_TRY(gemm_tn(dcur, W, sv.enc, IC, grads->pts_w[l], Kl, M, W, IC, st));
        NB_TRY(gemm_tn(dcur, W, hprev, W, grads->pts_w[l] + off, Kl, M, W, W, st));
        NB_TRY(gemm_nn(dcur, W, net->pts_w[l] + off, Kl, dnext, W, M, W, W, 0, st));
        float* t = dcur; dcur = dnext; dnext = t;
      }
    }
  }
  return 0;
}

// ---- tensor-core backward of one pass (bwd_tc2.cuh) ------------------------------------------------
namespace {
struct BwdTcLayout { size_t off_amax, off_draw, off_encv, off_dsum, off_gv, off_partial, off_grad, total; long long part_floats; };
struct BwdTcJobs { int n; WgradJob w[WG2_MAX_JOBS]; ReduceJob r[WG2_MAX_JOBS]; int total_ctas; long long part_floats; };

// jobs of the weight gradient and their CTA ranges (proportional to the bytes each job streams per tile)
BwdTcJobs make_bwd_jobs(const NerfNetParams& n, const NerfNetGrads* g, int sms) {
  BwdTcJobs J;
  memset(&J, 0, sizeof(J));
  const int D = n.D, W = n.W, IC = n.input_ch;
  auto add = [&](uint32_t a_off, int Mc, uint32_t b_off, int Nc, float* dst, int ldw, int n_valid, float* db) {
    WgradJob& w = J.w[J.n];
    ReduceJob& r = J.r[J.n];
    w.a_off = a_off; w.b_off = b_off; w.Mc = Mc; w.Nc = Nc; w.db = db; w.aux = 0; w.aux_dst = nullptr; w.aux_b = nullptr;
    r.Mc = Mc; r.Nc = Nc; r.n_valid = n_valid; r.ldw = ldw; r.dst = dst;
    ++J.n;
  };
  // job 0: G = d_hv^T h_{D-1} (-> views_linears[0].weight[:, :W] through views_feat_wgrad_kernel; its reduce target is a scratch
  // block set by the caller);  job 1: feature_linear = d_feat^T h_{D-1}
  add(0, 128, rec_act_h(D - 1), 256, nullptr, 256, 256, g ? g->views_b : nullptr);
  add(rec_grad_step(0), 256, rec_act_h(D - 1), 256, g ? g->feature_w : nullptr, W, W, g ? g->feature_b : nullptr);
  for (int l = D - 1; l >= 1; --l) {
    const bool sk = (n.skip >= 0 && l == n.skip + 1);
    add(rec_grad_dA(l, D), 256, rec_act_h(l - 1), 256, g ? g->pts_w[l] + (sk ? IC : 0) : nullptr, sk ? W + IC : W, W, g ? g->pts_b[l] : nullptr);
    if (sk) add(rec_grad_dA(l, D), 256, 0, 64, g ? g->pts_w[l] : nullptr, W + IC, IC, nullptr);        // the [input_pts] columns
  }
  add(rec_grad_dA(0, D), 256, 0, 64, g ? g->pts_w[0] : nullptr, IC, IC, g ? g->pts_b[0] : nullptr);
  // CTAs per job ~ its measured cost (profiles/r02_backward_experiments.txt: per-job finish times of a byte-proportional split):
  // bytes streamed per tile (Mc + Nc columns), x 1.27 for the feature job (its spare warps also sweep B for alpha_linear),
  // x 1.06 for the views job (per-ray atomics), x 1.16 for a 64-wide B with a bias gradient (short stages, same column sums)
  auto cost = [&](int i) {
    double c = (double)(J.w[i].Mc + J.w[i].Nc);
    if (i == 0) c *= 1.06;
    if (i == 1) c *= 1.27;
    if (J.w[i].Nc == 64 && J.w[i].db) c *= 1.16;
    return c;
  };
  double tot = 0;
  for (int i = 0; i < J.n; ++i) tot += cost(i);
  int used = 0;
  double frac[WG2_MAX_JOBS];
  for (int i = 0; i < J.n; ++i) {
    const double x = (double)sms * cost(i) / tot;
    int c = (int)x;
    if (c < 1) c = 1;
    frac[i] = x - c;
    J.w[i].ncta = c;
    used += c;
  }
  while (used < sms) {                               // leftovers: largest remainder first
    int b = 0;
    for (int i = 1; i < J.n; ++i) if (frac[i] > frac[b]) b = i;
    ++J.w[b].ncta; ++used; frac[b] -= 1.0;
  }
  while (used > sms) {                               // (only where the GPU has few SMs for the number of jobs)
    int b = 0;
    for (int i = 1; i < J.n; ++i) if (J.w[i].ncta > J.w[b].ncta) b = i;
    --J.w[b].ncta; --used;
  }
  int cta = 0;
  long long pf = 0;
  for (int i = 0; i < J.n; ++i) {
    J.w[i].cta0 = cta; cta += J.w[i].ncta;
    J.w[i].part_off = pf; J.r[i].part_off = pf; J.r[i].ncta = J.w[i].ncta;
    pf += (long long)J.w[i].ncta * J.w[i].Mc * J.w[i].Nc;
  }
  J.total_ctas = cta; J.part_floats = pf;
  return J;
}

BwdTcLayout make_bwd_layout(long long N, int S, const NerfNetParams& n, const TilePlan& plan, long long part_floats) {
  BwdTcLayout L;
  auto up = [](size_t x) { return (x + 1023) & ~(size_t)1023; };
  size_t o = 0;
  L.off_amax = o;    o = up(o + 256);
  L.off_draw = o;    o = up(o + (size_t)N * S * 16);
  L.off_encv = o;    o = up(o + (size_t)N * (n.input_ch_views > 0 ? n.input_ch_views : 1) * 4);
  L.off_dsum = o;    o = up(o + (size_t)N * 128 * 4);
  L.off_gv = o;      o = up(o + (size_t)(128 * 256 + 128) * 4);      // G = d_hv^T h_{D-1} (reduced) and this pass's db_v
  L.off_partial = o; o = up(o + (size_t)part_floats * 4);
  L.off_grad = o;    o = up(o + (size_t)plan.n_tiles * rec_grad_bytes(n.D));
  L.total = o; L.part_floats = part_floats;
  return L;
}
}  // namespace

static size_t bwd_pass_bytes(int64_t N, int S, const NerfNetParams* net) {
  const int sms = num_sms();
  const TilePlan plan = make_tile_plan(N, S, sms);
  return make_bwd_layout(N, S, *net, plan, (long long)sms * 256 * 256).total + 1024;
}

size_t nerf_b200_march_bwd_tc_workspace_bytes(int64_t N, int S, const NerfNetParams* net) {
  if (!net || check_tc_net(net) || !net->use_viewdirs || N <= 0 || S <= 0) return 0;
  return bwd_pass_bytes(N, S, net);
}

// introspection for tests and tools: where nerf_b200_march_bwd_tc keeps its intermediates inside the (1 KB-aligned)
// workspace and how the tiles are laid out.  out[0..11] = off_d_raw, off_grad_records, rec_act_bytes, rec_mask_bytes,
// rec_grad_bytes, grid, rays_per_cta, nst, n_tiles, off_amax, off_dsum, off_partial
int nerf_b200_march_bwd_tc_layout(int64_t N, int S, const NerfNetParams* net, int64_t* out) {
  if (int rc = check_tc_net(net)) return rc;
  NB_CHECK_ARG(out && N > 0 && S > 0 && net->use_viewdirs, "bad arguments");
  const int sms = num_sms();
  const TilePlan plan = make_tile_plan(N, S, sms);
  const BwdTcLayout LY = make_bwd_layout(N, S, *net, plan, (long long)sms * 256 * 256);
  out[0] = (int64_t)LY.off_draw; out[1] = (int64_t)LY.off_grad; out[2] = rec_act_bytes(net->D); out[3] = rec_mask_bytes(net->D);
  out[4] = rec_grad_bytes(net->D); out[5] = plan.grid; out[6] = plan.rays_per_cta; out[7] = plan.nst; out[8] = plan.n_tiles;
  out[9] = (int64_t)LY.off_amax; out[10] = (int64_t)LY.off_dsum; out[11] = (int64_t)LY.off_partial;
  return 0;
}

namespace {
// One pass of the tensor-core backward, split into its phases so that the two passes of render_rays can interleave: the small
// kernels of one pass (prologue, heads) run on a side stream next to the other pass's big kernels (dgrad, wgrad), which each
// take the whole GPU.  run() is the pass on one stream.
struct BwdTcPass {
  const float* rays; const float* z; const float* noise; int64_t N; int S; const NerfNetParams* net; const void* packed;
  const NerfRenderCfg* cfg; const float* raw; const NerfTrainSave* save; const float* g_rgb; const NerfNetGrads* grads;
  DeviceState* ds; TilePlan plan; BwdTcLayout LY; PackLayout PL;
  unsigned int* amax; float *d_raw, *encv, *dsum, *gv, *dbv, *partial; uint8_t* grec; const uint8_t *act, *mask;

  int init(void* workspace, size_t workspace_bytes) {
    ds = device_state();
    plan = make_tile_plan(N, S, ds->sms);
    LY = make_bwd_layout(N, S, *net, plan, (long long)ds->sms * 256 * 256);
    uint8_t* ws = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(workspace) + 1023) & ~(uintptr_t)1023);
    NB_CHECK_ARG(workspace && workspace_bytes >= LY.total + (size_t)(ws - static_cast<uint8_t*>(workspace)), "march_bwd_tc workspace too small (%zu < %zu)", workspace_bytes, LY.total + 1024);
    NB_CHECK_ARG(save->act && save->mask && save->act_bytes >= (size_t)plan.n_tiles * rec_act_bytes(net->D) && save->mask_bytes >= (size_t)plan.n_tiles * rec_mask_bytes(net->D),
                 "training-mode records missing or too small");
    PL = make_pack_layout(*net);
    amax = reinterpret_cast<unsigned int*>(ws + LY.off_amax);
    d_raw = reinterpret_cast<float*>(ws + LY.off_draw);
    encv = reinterpret_cast<float*>(ws + LY.off_encv);
    dsum = reinterpret_cast<float*>(ws + LY.off_dsum);
    gv = reinterpret_cast<float*>(ws + LY.off_gv);
    dbv = gv + 128 * 256;
    partial = reinterpret_cast<float*>(ws + LY.off_partial);
    grec = ws + LY.off_grad;
    act = static_cast<const uint8_t*>(save->act);
    mask = static_cast<const uint8_t*>(save->mask);
    if (!ds->optin_bwd) {
      NB_TRY(smem_optin((const void*)dgrad_tc2_kernel, SM_ALLOC));
      NB_TRY(smem_optin((const void*)wgrad_tc_kernel, WG2_TOTAL));
      ds->optin_bwd = true;
    }
    return 0;
  }

  // 1. loss scale from max |dL/drgb_map|; compositing adjoint -> dL/draw (SURVEY App. E);  2. seed of the chain: d_hv tiles
  int prologue(cudaStream_t st) {
    const int sms = ds->sms, D = net->D;
    NB_CUDA(cudaMemsetAsync(amax, 0, 256, st));
    NB_CUDA(cudaMemsetAsync(dsum, 0, (size_t)N * 128 * 4, st));
    NB_CUDA(cudaMemsetAsync(gv, 0, (size_t)(128 * 256 + 128) * 4, st));
    absmax_kernel<<<cdiv(N * 3, 1024) < 64 ? cdiv(N * 3, 1024) : 64, 256, 0, st>>>(g_rgb, N * 3, amax);
    NB_LAUNCH_OK("absmax_kernel");
    NB_TRY(nerf_b200_raw2outputs_bwd(raw, z, rays + 3, cfg->ray_stride, noise, N, S, cfg->white_bkgd, g_rgb, d_raw, (void*)st));
    SeedParams sp;
    sp.d_raw = d_raw; sp.mask = mask; sp.act = act; sp.grad = grec; sp.rgb_w = net->rgb_w; sp.amax = amax;
    sp.N = N; sp.S = S; sp.rays_per_cta = plan.rays_per_cta; sp.nst_plan = plan.nst; sp.D = D;
    sp.rec_mask = rec_mask_bytes(D); sp.rec_act = rec_act_bytes(D); sp.rec_grad = rec_grad_bytes(D); sp.n_tiles = plan.n_tiles;
    sp.g_rgb_w = grads->rgb_w; sp.g_rgb_b = grads->rgb_b;
    dhv_seed_heads_kernel<<<(int)(plan.n_tiles < 3 * sms ? plan.n_tiles : 3 * sms), 256, 0, st>>>(sp);
    NB_LAUNCH_OK("dhv_seed_heads_kernel");
    return 0;
  }

  // 3. dgrad chain: the forward's grid (CTA pairs), CTA b serves the tiles of forward CTA b
  int dgrad(cudaStream_t st) {
    const int D = net->D;
    const uint8_t* pk = static_cast<const uint8_t*>(packed);
    DgradParams dp;
    dp.mask = mask; dp.grad = grec; dp.d_raw = d_raw; dp.amax = amax; dp.alpha_w = net->alpha_w;
    dp.N = N; dp.S = S; dp.rays_per_cta = plan.rays_per_cta; dp.nst_plan = plan.nst; dp.D = D;
    dp.rec_mask = rec_mask_bytes(D); dp.rec_grad = rec_grad_bytes(D);
    dp.pair_half_bytes = PL.bwd_bytes / 2;
    CUtensorMap wmap, gmap;
    NB_TRY(make_row_map(&wmap, pk + PL.off_bwd_pair, PL.bwd_bytes, 16));
    NB_TRY(make_row_map(&gmap, grec, (size_t)plan.n_tiles * rec_grad_bytes(D), 16));      // 8 KB boxes: the pieces of the d_hv image
    TimedLaunch* tl = nullptr;
    if (g_timing && g_ntimed < 4096) {
      tl = &g_timed[g_ntimed++];
      cudaEventCreate(&tl->a); cudaEventCreate(&tl->b);
      tl->flops = 2.0 * ((double)(net->W / 2) * net->W + (double)D * net->W * net->W) * (double)(N * (long long)S);
      tl->kind = 1;
      cudaEventRecord(tl->a, st);
    }
    dgrad_tc2_kernel<<<plan.grid, TC_THREADS, SM_ALLOC, st>>>(dp, wmap, gmap);
    if (tl) cudaEventRecord(tl->b, st);
    NB_LAUNCH_OK("dgrad_tc2_kernel");
    return 0;
  }

  // 4. weight gradients (layer-major) + bias gradients on all SMs, then the reduction of the per-CTA partial blocks (adds
  // into the gradient tensors)
  int wgrad(cudaStream_t st) {
    const int D = net->D;
    BwdTcJobs J = make_bwd_jobs(*net, grads, ds->sms & ~1);        // whole CTA pairs: the kernel launches as 2-CTA clusters
    J.w[0].aux = 1; J.w[0].aux_dst = dsum;            // views job: per-ray row sums of d_hv
    J.w[1].aux = 2; J.w[1].aux_dst = grads->alpha_w; J.w[1].aux_b = grads->alpha_b;   // feature job: alpha_linear gradients
    WgradParams wp;
    memset(&wp, 0, sizeof(wp));
    wp.act = act; wp.grad = grec; wp.rec_act = rec_act_bytes(D); wp.rec_grad = rec_grad_bytes(D);
    wp.N = N; wp.S = S; wp.rays_per_cta = plan.rays_per_cta; wp.nst_plan = plan.nst; wp.n_tiles = plan.n_tiles;
    wp.amax = amax; wp.partial = partial; wp.d_raw = d_raw; wp.njobs = J.n;
    for (int i = 0; i < J.n; ++i) wp.jobs[i] = J.w[i];
    TimedLaunch* tl = nullptr;
    if (g_timing && g_ntimed < 4096) {
      tl = &g_timed[g_ntimed++];
      cudaEventCreate(&tl->a); cudaEventCreate(&tl->b);
      tl->flops = 2.0 * (net_macs_per_row(*net) - (double)net->W - 3.0 * (net->W / 2) - (double)net->input_ch_views * (net->W / 2)) * (double)(N * (long long)S);
      tl->kind = 2;
      cudaEventRecord(tl->a, st);
    }
    wgrad_tc_kernel<<<J.total_ctas, WG2_THREADS, WG2_TOTAL, st>>>(wp);
    if (tl) cudaEventRecord(tl->b, st);
    NB_LAUNCH_OK("wgrad_tc_kernel");
    ReduceParams rp;
    memset(&rp, 0, sizeof(rp));
    rp.partial = partial; rp.amax = amax; rp.njobs = J.n;
    J.r[0].dst = gv;                                  // job 0 reduces into the scratch block G
    for (int i = 0; i < J.n; ++i) rp.jobs[i] = J.r[i];
    dim3 rg(256, J.n);
    wgrad_reduce_kernel<<<rg, 256, 0, st>>>(rp);
    NB_LAUNCH_OK("wgrad_reduce_kernel");
    return 0;
  }

  // 5. the view columns of views_linears[0] (after ALL of the pass's weight-gradient launches)
  int heads(cudaStream_t st) {
    const int ICV = net->input_ch_views;
    encv_kernel<<<cdiv(N * ICV, 256), 256, 0, st>>>(rays + 8, cfg->ray_stride, N, ICV, encv);
    NB_LAUNCH_OK("encv_kernel");
    dim3 vg(ICV + 1, cdiv(N, 64));
    views_enc_wgrad_kernel<<<vg, 128, 0, st>>>(dsum, encv, N, ICV, grads->views_w, net->W + ICV, net->W, dbv);
    NB_LAUNCH_OK("views_enc_wgrad_kernel");
    views_feat_wgrad_kernel<<<128, 256, 0, st>>>(gv, dbv, net->feature_w, net->feature_b, grads->views_w, net->W + ICV);
    NB_LAUNCH_OK("views_feat_wgrad_kernel");
    return 0;
  }

  // the whole pass on one stream
  int run(cudaStream_t st) {
    NB_TRY(prologue(st));
    NB_TRY(dgrad(st));
    NB_TRY(wgrad(st));
    return heads(st);
  }
};

int check_bwd_pass(const float* rays, const NerfBwdPass* q, const NerfRenderCfg* cfg) {
  NB_CHECK_ARG(rays && q && q->z_vals && q->net && q->packed && cfg && q->raw && q->save && q->g_rgb && q->grads, "NULL pointer");
  if (int rc = check_tc_net(q->net)) return rc;
  NB_CHECK_ARG(q->net->use_viewdirs, "the tensor-core backward serves use_viewdirs networks (exact mode serves the others)");
  NB_CHECK_ARG(q->net->W == 256, "the tensor-core backward supports netwidth == 256");
  NB_CHECK_ARG(q->S > 0, "S must be positive");
  return 0;
}
BwdTcPass bind_pass(const float* rays, int64_t N, const NerfRenderCfg* cfg, const NerfBwdPass* q) {
  BwdTcPass b;
  memset(&b, 0, sizeof(b));
  b.rays = rays; b.z = q->z_vals; b.noise = q->noise; b.N = N; b.S = q->S; b.net = q->net; b.packed = q->packed; b.cfg = cfg;
  b.raw = q->raw; b.save = q->save; b.g_rgb = q->g_rgb; b.grads = q->grads;
  return b;
}
}  // namespace

int nerf_b200_march_bwd_tc(const float* rays, const float* z_vals, const float* noise, int64_t N, int S, const NerfNetParams* net,
                           const void* packed, const NerfRenderCfg* cfg, const float* raw, const NerfTrainSave* save,
                           const float* g_rgb, const NerfNetGrads* grads, void* workspace, size_t workspace_bytes, void* stream) {
  NerfBwdPass q;
  q.z_vals = z_vals; q.noise = noise; q.S = S; q.net = net; q.packed = packed; q.raw = raw; q.save = save; q.g_rgb = g_rgb; q.grads = grads;
  if (int rc = check_bwd_pass(rays, &q, cfg)) return rc;
  if (N == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  BwdTcPass b = bind_pass(rays, N, cfg, &q);
  NB_TRY(b.init(workspace, workspace_bytes));
  return b.run(st);
}

size_t nerf_b200_render_rays_bwd_tc_workspace_bytes(int64_t N, int S_coarse, const NerfNetParams* net_coarse, int S_fine, const NerfNetParams* net_fine) {
  if (!net_coarse || check_tc_net(net_coarse) || !net_coarse->use_viewdirs || N <= 0 || S_coarse <= 0) return 0;
  size_t b = bwd_pass_bytes(N, S_coarse, net_coarse);
  if (net_fine && S_fine > 0) {
    if (check_tc_net(net_fine) || !net_fine->use_viewdirs) return 0;
    b += bwd_pass_bytes(N, S_fine, net_fine);
  }
  return b;
}

// Backward of both passes of render_rays (run_nerf.py:765-772: loss = img2mse(rgb) + img2mse(rgb0); z_samples is detached, :394,
// so the passes are independent).  Two streams (graph-capturable: the side stream forks from and joins `stream`):
//   main: prologue(c) dgrad(c) | wgrad(c)      | dgrad(f) | wgrad(f) heads(f) |
//   side:                      | prologue(f)   |          | heads(c)          | join
// the small memory-bound kernels of one pass (compositing adjoint, seed tiles + rgb_linear, view-column gradients) run on the SM
// resources the weight-gradient kernel leaves free (it holds one 192-thread CTA per SM) instead of between the big kernels.
// One stream, one pass after the other: a single pass, one network serving both passes (its gradients would race), a fine
// pass of fewer than 4 CTAs, or no side stream (its creation failed).
int nerf_b200_render_rays_bwd_tc(const float* rays, int64_t N, const NerfRenderCfg* cfg, const NerfBwdPass* coarse, const NerfBwdPass* fine,
                                 void* workspace, size_t workspace_bytes, void* stream) {
  if (int rc = check_bwd_pass(rays, coarse, cfg)) return rc;
  if (fine) if (int rc = check_bwd_pass(rays, fine, cfg)) return rc;
  if (N == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  BwdTcPass c = bind_pass(rays, N, cfg, coarse);
  const size_t cb = bwd_pass_bytes(N, coarse->S, coarse->net);
  NB_CHECK_ARG(workspace && workspace_bytes >= cb, "render_rays_bwd_tc workspace too small");
  NB_TRY(c.init(workspace, cb));
  if (!fine) return c.run(st);
  BwdTcPass f = bind_pass(rays, N, cfg, fine);
  NB_TRY(f.init(static_cast<uint8_t*>(workspace) + cb, workspace_bytes - cb));
  DeviceState* ds = c.ds;
  const bool shared_grads = (coarse->grads->pts_w[0] == fine->grads->pts_w[0]);
  if (shared_grads || f.plan.grid < 4 || !ds->side) {
    NB_TRY(c.run(st));
    return f.run(st);
  }
  cudaStream_t sd = ds->side;
  NB_TRY(c.prologue(st));
  NB_TRY(c.dgrad(st));
  NB_CUDA(cudaEventRecord(ds->ev[0], st));
  NB_CUDA(cudaStreamWaitEvent(sd, ds->ev[0], 0));
  NB_TRY(f.prologue(sd));
  NB_CUDA(cudaEventRecord(ds->ev[1], sd));
  NB_TRY(c.wgrad(st));
  NB_CUDA(cudaStreamWaitEvent(st, ds->ev[1], 0));
  NB_TRY(f.dgrad(st));
  NB_CUDA(cudaEventRecord(ds->ev[2], st));
  NB_CUDA(cudaStreamWaitEvent(sd, ds->ev[2], 0));
  NB_TRY(c.heads(sd));
  NB_CUDA(cudaEventRecord(ds->ev[3], sd));
  NB_TRY(f.wgrad(st));
  NB_TRY(f.heads(st));
  NB_CUDA(cudaStreamWaitEvent(st, ds->ev[3], 0));
  return 0;
}

// ---- the two ends of the optimisation step (train_step.cuh) ------------------------------------------
int nerf_b200_mse_seed(const float* rgb, const float* target, int64_t N, float grad_scale, float* g_rgb, float* loss_accum, void* stream) {
  NB_CHECK_ARG(rgb && target && g_rgb && loss_accum, "NULL pointer");
  if (N == 0) return 0;
  const long long n3 = N * 3;
  mse_seed_kernel<<<cdiv(n3, 256) < 64 ? cdiv(n3, 256) : 64, 256, 0, (cudaStream_t)stream>>>(rgb, target, n3, 1.0f / (float)n3, grad_scale, g_rgb, loss_accum);
  NB_LAUNCH_OK("mse_seed_kernel");
  return 0;
}

int nerf_b200_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n, float* state,
                        float lr0, float decay_rate, float decay_steps, float beta1, float beta2, float eps, float grad_mul, void* stream) {
  NB_CHECK_ARG(params && grads && exp_avg && exp_avg_sq && state, "NULL pointer");
  if (n == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  const int grid = cdiv(n, 1024) < 4 * num_sms() ? cdiv(n, 1024) : 4 * num_sms();
  adam_flat_kernel<<<grid, 256, 0, st>>>(params, grads, exp_avg, exp_avg_sq, n, state, lr0, decay_rate, decay_steps, beta1, beta2, eps, grad_mul);
  NB_LAUNCH_OK("adam_flat_kernel");
  adam_advance_kernel<<<1, 1, 0, st>>>(state, lr0, decay_rate, decay_steps);
  NB_LAUNCH_OK("adam_advance_kernel");
  return 0;
}

}  // extern "C"
