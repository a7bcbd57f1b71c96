/*
 * nerf_b200.h -- C ABI of the B200-native NeRF ray-marching hot path.
 *
 * Drop-in boundary for yenchenlin/nerf-pytorch's  render_rays -> run_network/batchify ->
 * NeRF.forward -> raw2outputs  (+ sample_pdf, Embedder).  The reference has no FFI of its own
 * (it is pure Python on torch); each entry point below names the reference function (file:line
 * under /root/reference) whose tensor-op chain it replaces.  Conventions:
 *
 *   - every pointer is a DEVICE pointer to fp32 data owned by the caller (torch), borrowed for
 *     the duration of the call; outputs and workspaces are caller-allocated;
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream); no call
 *     synchronises the device or the stream;
 *   - return value 0 = OK, negative = error; nerf_b200_last_error() gives the message
 *     (thread-local).  The Python host turns a non-zero return into RuntimeError, which is the
 *     reference's only error convention (Python exceptions);
 *   - no CPU fallback exists: every entry point launches sm_100a kernels.
 */
#ifndef NERF_B200_H_
#define NERF_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NERF_B200_ABI_VERSION 1
#define NERF_B200_MAX_D 16

/* Live parameter storages of one reference `NeRF` module (run_nerf_helpers.py:67-94):
 * nn.Linear layout, weight [out,in] row-major fp32, bias [out].  Unused pointers are NULL. */
typedef struct NerfNetParams {
  int32_t D;               /* number of pts_linears (netdepth, 8)                               */
  int32_t W;               /* hidden width (netwidth, 256)                                     */
  int32_t input_ch;        /* encoded point channels (63)                                      */
  int32_t input_ch_views;  /* encoded view channels (27), 0 when !use_viewdirs                 */
  int32_t skip;            /* layer index after which [input_pts, h] is concatenated (4), -1 = none */
  int32_t use_viewdirs;    /* 1: alpha/feature/views/rgb heads; 0: output_linear               */
  int32_t output_ch;       /* rows of output_linear when !use_viewdirs (4 or 5)                */
  int32_t reserved;
  const float* pts_w[NERF_B200_MAX_D];   /* pts_linears.i.weight                                */
  const float* pts_b[NERF_B200_MAX_D];   /* pts_linears.i.bias                                  */
  const float* feature_w; const float* feature_b;   /* feature_linear  [W,W]                   */
  const float* alpha_w;   const float* alpha_b;     /* alpha_linear    [1,W]                   */
  const float* views_w;   const float* views_b;     /* views_linears.0 [W/2, W+input_ch_views] */
  const float* rgb_w;     const float* rgb_b;       /* rgb_linear      [3,W/2]                 */
  const float* output_w;  const float* output_b;    /* output_linear   [output_ch,W]           */
} NerfNetParams;

/* Static configuration of one render_rays call (run_nerf.py:308-320 keyword arguments). */
typedef struct NerfRenderCfg {
  int32_t N_samples;       /* coarse samples per ray (64)                                      */
  int32_t N_importance;    /* extra fine samples per ray (0 / 64 / 128)                        */
  int32_t multires;        /* L for points (10)  -> 3+6L channels                              */
  int32_t multires_views;  /* L for view dirs (4)                                              */
  int32_t lindisp;         /* run_nerf.py:361                                                  */
  int32_t perturb;         /* 1: z = lower + (upper-lower)*t_rand (run_nerf.py:365-379)        */
  int32_t white_bkgd;      /* run_nerf.py:302-303                                              */
  int32_t ray_stride;      /* floats per ray row: 11 (o,d,near,far,viewdir) or 8               */
  int32_t precision;       /* NERF_B200_PREC_*                                                 */
  int32_t reserved[3];
} NerfRenderCfg;

#define NERF_B200_PREC_TC_FP16 0   /* tcgen05 kind::f16, fp16 operands, fp32 accumulate (fast path) */
#define NERF_B200_PREC_FP32    1   /* CUDA-core fp32 FMA chain (exact mode, validation)             */

/* Outputs of one network pass over N rays x S samples.  NULL pointers are skipped. */
typedef struct NerfPassOut {
  float* rgb_map;   /* [N,3]            run_nerf.py:296,303 */
  float* disp_map;  /* [N]              run_nerf.py:299     */
  float* acc_map;   /* [N]              run_nerf.py:300     */
  float* depth_map; /* [N]              run_nerf.py:298     */
  float* weights;   /* [N,S]            run_nerf.py:295     */
  float* raw;       /* [N,S,4] rgb,sigma  (retraw, run_nerf.py:406-407) */
} NerfPassOut;

int         nerf_b200_abi_version(void);
const char* nerf_b200_last_error(void);

/* ---- Embedder.embed (run_nerf_helpers.py:36-45): x [M,3] -> out [M, 3+6L] ------------------- */
int nerf_b200_embed(const float* x, int64_t M, int L, float* out, void* stream);

/* ---- weight packing: fp32 nn.Linear storages -> fp16 UMMA-swizzled chunk stream + fp32 heads -- */
/* (replaces nothing in the reference; it is the analogue of `.to(device)` at run_nerf.py:191)     */
size_t nerf_b200_packed_bytes(const NerfNetParams* net);
int    nerf_b200_pack_weights(const NerfNetParams* net, void* packed, size_t packed_bytes, void* stream);

/* ---- run_network + batchify + NeRF.forward (run_nerf.py:27-51, run_nerf_helpers.py:96-119) --- */
/* pts [N*S,3], viewdirs [N,3] (NULL when the net has no view input) -> raw [N*S,4].               */
/* precision TC_FP16 needs `packed` (from nerf_b200_pack_weights); FP32 needs `net`.               */
int nerf_b200_run_network(const float* pts, const float* viewdirs, int64_t N, int S,
                          const NerfNetParams* net, const void* packed, int multires,
                          int multires_views, int precision, float* raw,
                          void* workspace, size_t workspace_bytes, void* stream);

/* ---- raw2outputs (run_nerf.py:262-305) and its adjoint (SURVEY App. E) ------------------------ */
/* raw [N,S,4], z_vals [N,S], rays_d row pointer with stride `d_stride` floats, noise [N,S]|NULL.  */
int nerf_b200_raw2outputs(const float* raw, const float* z_vals, const float* rays_d, int d_stride,
                          const float* noise, int64_t N, int S, int white_bkgd,
                          const NerfPassOut* out, void* stream);
int nerf_b200_raw2outputs_bwd(const float* raw, const float* z_vals, const float* rays_d, int d_stride,
                              const float* noise, int64_t N, int S, int white_bkgd,
                              const float* g_rgb /*[N,3]*/, float* d_raw /*[N,S,4]*/, void* stream);

/* ---- sample_pdf (run_nerf_helpers.py:196-239): bins [N,B], weights [N,B-1], u [N or 1, n_samples]
 *      (u_row_stride 0 = the det linspace row shared by all rays) -> samples [N,n_samples] ------- */
int nerf_b200_sample_pdf(const float* bins, const float* weights, const float* u, int64_t u_row_stride,
                         int64_t N, int B, int n_samples, float* samples, void* stream);

/* ---- z sampling of render_rays (run_nerf.py:357-379): rays [N,ray_stride], t_vals [S] (the
 *      torch.linspace row), t_rand [N,S]|NULL -> z_vals [N,S] ------------------------------------ */
int nerf_b200_coarse_z(const float* rays, int ray_stride, const float* t_vals, const float* t_rand,
                       int64_t N, int S, int lindisp, float* z_vals, void* stream);

/* ---- ray batch construction of render() (run_nerf.py:95-123): optional pinhole ray generation (get_rays,
 *      run_nerf_helpers.py:153-162) for pixels [pixel0, pixel0+N) of an H x W image, view-direction
 *      normalisation (:108), optional NDC warp (ndc_rays, run_nerf_helpers.py:175-192, near plane 1) and packing
 *      to out [N, 11 | 8] = o(3) d(3) near far [viewdir(3)].  rays_o/rays_d [N,3] or both NULL (generate from
 *      `cam`); view_src [N,3] = directions to normalise into viewdirs (NULL -> rays_d, as in :104). ----------- */
typedef struct NerfCamera {
  int32_t H, W;
  float fx, fy, cx, cy;      /* K[0][0], K[1][1], K[0][2], K[1][2] (run_nerf.py:615-620) */
  float c2w[12];             /* camera-to-world [3,4], row-major */
} NerfCamera;
int nerf_b200_pack_rays(const float* rays_o, const float* rays_d, const float* view_src, const NerfCamera* cam,
                        int64_t N, int64_t pixel0, int ndc, float near, float far, int use_viewdirs,
                        float* out, void* stream);
/* the arguments of nerf_b200_pack_rays as a struct: nerf_b200_render_fwd builds the batch inside its per-ray prologue launch */
typedef struct NerfRayGen {
  const float* rays_o; const float* rays_d;   /* [N,3] each, or both NULL: generate from `cam` for pixels [pixel0, pixel0 + N) */
  const float* view_src;                      /* [N,3] or NULL */
  const NerfCamera* cam;                      /* needed to generate rays and for ndc */
  int64_t pixel0;
  int32_t ndc, use_viewdirs;
  float near, far;
} NerfRayGen;
/* same, for an arbitrary device list of pixel ids (row-major j * W + i) of the camera's image: the per-image random
 * pixel choice of train() (run_nerf.py:728-757: get_rays for the whole image, meshgrid, np.random.choice, gather)
 * without the [H,W,3] ray tensors (SURVEY 8f rank 3) */
int nerf_b200_pack_rays_pixels(const NerfCamera* cam, const int64_t* pixel_index, int64_t N, int ndc, float near,
                               float far, int use_viewdirs, float* out, void* stream);
/* to8b (run_nerf_helpers.py:11) on the device: out[i] = uint8(255 * clip(x[i], 0, 1)) -- image output of render_path
 * (run_nerf.py:160-169) without a float32 round trip through the host */
int nerf_b200_to8b(const float* x, int64_t n, uint8_t* out, void* stream);

/* ---- hierarchical resampling of render_rays (run_nerf.py:392-396, :412): z_mid, sample_pdf on
 *      weights[...,1:-1], sort(cat) and z_std in one kernel.
 *      z_vals [N,S], weights [N,S], u as above -> z_fine [N,S+n_imp] sorted, z_std [N] ------------ */
int nerf_b200_fine_z(const float* z_vals, const float* weights, const float* u, int64_t u_row_stride,
                     int64_t N, int S, int n_imp, float* z_fine, float* z_samples /*[N,n_imp]|NULL*/,
                     float* z_std, void* stream);

/* ---- one fused network pass: pts = o + d*z  -> encode -> MLP (tcgen05) -> raw2outputs ----------
 *      replaces run_nerf.py:381-386 (coarse) / :397-403 (fine).  rays [N,ray_stride], z_vals [N,S],
 *      noise [N,S]|NULL.  sigma/rgb stay on chip unless out->raw is requested. -------------------- */
int nerf_b200_march(const float* rays, const float* z_vals, const float* noise, int64_t N, int S,
                    const NerfNetParams* net, const void* packed, const NerfRenderCfg* cfg,
                    const NerfPassOut* out, void* workspace, size_t workspace_bytes, void* stream);
size_t nerf_b200_march_workspace_bytes(int64_t N, int S);

/* ---- whole render_rays forward (run_nerf.py:308-418) for one ray chunk -------------------------
 *      t_vals [N_samples] / u_det [N_importance]: the torch.linspace rows; t_rand, u_rand, noise0,
 *      noise1: injected RNG draws or NULL.  coarse/fine: outputs of the two passes (fine may be
 *      NULL when N_importance == 0).  z_fine/z_std: [N,S_c+N_imp] / [N] (required when
 *      N_importance > 0). ------------------------------------------------------------------------ */
int nerf_b200_render_rays_fwd(const float* rays, int64_t N, const NerfRenderCfg* cfg,
                              const NerfNetParams* net_coarse, const void* packed_coarse,
                              const NerfNetParams* net_fine, const void* packed_fine,
                              const float* t_vals, const float* u_det,
                              const float* t_rand, const float* u_rand,
                              const float* noise0, const float* noise1,
                              float* z_coarse /*[N,S_c]*/, const NerfPassOut* coarse,
                              float* z_fine, float* z_std, const NerfPassOut* fine,
                              void* workspace, size_t workspace_bytes, void* stream);
/* render() for one chunk (run_nerf.py:69-134 with N <= chunk): nerf_b200_render_rays_fwd whose prologue launch also BUILDS the ray
 * batch `rays` [N, 8 | 11] from `gen` (one launch less than pack_rays + render_rays_fwd; the exact path launches pack_rays itself) */
int nerf_b200_render_fwd(const NerfRayGen* gen, float* rays, int64_t N, const NerfRenderCfg* cfg,
                         const NerfNetParams* net_coarse, const void* packed_coarse, const NerfNetParams* net_fine,
                         const void* packed_fine, const float* t_vals, const float* u_det, const float* t_rand,
                         const float* u_rand, const float* noise0, const float* noise1, float* z_coarse,
                         const NerfPassOut* coarse, float* z_fine, float* z_std, const NerfPassOut* fine,
                         void* workspace, size_t workspace_bytes, void* stream);

/* ---- training mode of the fused pass: besides its outputs (out->raw is required) the pass leaves, per 128-row
 *      tile, a record of fp16 activation images (encodings, post-ReLU h_l, view layer; 560 KB for D = 8) and the
 *      sign bits of the pre-activations (csrc/train_common.cuh) -- what the reference's autograd saves
 *      (run_nerf_helpers.py:96-119), but written once, in the MMA operand layout (two 64-row half images per
 *      tile image), by cp.async.bulk from the shared-memory tiles the forward produces anyway.
 *      use_viewdirs networks, tensor-core precision. ---------------------------------------------------------- */
typedef struct NerfTrainSave {
  void*  act;   size_t act_bytes;    /* activation records: nerf_b200_train_record_bytes(...)            */
  void*  mask;  size_t mask_bytes;   /* ReLU sign-bit records                                            */
} NerfTrainSave;
int nerf_b200_train_record_bytes(int64_t N, int S, const NerfNetParams* net, size_t* act_bytes, size_t* mask_bytes);
int nerf_b200_march_train(const float* rays, const float* z_vals, const float* noise, int64_t N, int S,
                          const NerfNetParams* net, const void* packed, const NerfRenderCfg* cfg,
                          const NerfPassOut* out, void* workspace, size_t workspace_bytes,
                          const NerfTrainSave* save, void* stream);
/* nerf_b200_render_rays_fwd with both passes in training mode (the render call of run_nerf.py:760-762,
 * retraw=True): coarse->raw and fine->raw are required. */
int nerf_b200_render_rays_fwd_train(const float* rays, int64_t N, const NerfRenderCfg* cfg,
                                    const NerfNetParams* net_coarse, const void* packed_coarse,
                                    const NerfNetParams* net_fine, const void* packed_fine,
                                    const float* t_vals, const float* u_det,
                                    const float* t_rand, const float* u_rand,
                                    const float* noise0, const float* noise1,
                                    float* z_coarse, const NerfPassOut* coarse,
                                    float* z_fine, float* z_std, const NerfPassOut* fine,
                                    void* workspace, size_t workspace_bytes,
                                    const NerfTrainSave* save_coarse, const NerfTrainSave* save_fine, void* stream);

/* ---- backward of one network pass: what loss.backward() (run_nerf.py:775) does through
 *      run_nerf.py:381-386 / :397-403.  dL/dtheta is ACCUMULATED (+=) into fp32 grads laid out like the
 *      reference parameters; g_rgb [N,3] = dL/drgb_map (the only output the reference's loss reads,
 *      run_nerf.py:765-772); no gradient flows to rays or z (run_nerf.py:394). ---------------------------- */
typedef struct NerfNetGrads {
  float* pts_w[NERF_B200_MAX_D]; float* pts_b[NERF_B200_MAX_D];
  float* feature_w; float* feature_b; float* alpha_w; float* alpha_b;
  float* views_w;   float* views_b;   float* rgb_w;   float* rgb_b;
  float* output_w;  float* output_b;
} NerfNetGrads;
/* tensor-core backward (csrc/bwd_tc2.cuh): compositing adjoint, tcgen05 dgrad chain with loss-scaled fp16
 * activation gradients, layer-major tcgen05 weight gradient; consumes the records of the training-mode pass
 * and its raw [N,S,4]. */
int nerf_b200_march_bwd_tc(const float* rays, const float* z_vals, const float* noise, int64_t N, int S,
                           const NerfNetParams* net, const void* packed, const NerfRenderCfg* cfg,
                           const float* raw, const NerfTrainSave* save, const float* g_rgb,
                           const NerfNetGrads* grads, void* workspace, size_t workspace_bytes, void* stream);
size_t nerf_b200_march_bwd_tc_workspace_bytes(int64_t N, int S, const NerfNetParams* net);
/* introspection (tests / tools): offsets of the intermediates inside the 1 KB-aligned workspace and the tile plan:
 * out[12] = off_d_raw, off_grad_records, rec_act_bytes, rec_mask_bytes, rec_grad_bytes, grid, rays_per_cta, nst,
 * n_tiles, off_amax, off_dsum, off_partial */
int nerf_b200_march_bwd_tc_layout(int64_t N, int S, const NerfNetParams* net, int64_t* out);
/* Backward of BOTH passes of one render_rays call -- what loss.backward() triggers for loss = img2mse(rgb) + img2mse(rgb0)
 * (run_nerf.py:765-772; z_samples is detached at :394, so the two passes are independent).  Same kernels as
 * nerf_b200_march_bwd_tc per pass, but scheduled together: the data-gradient chain of one pass (HBM-write-bound) runs on
 * part of the SMs next to the weight gradient of the other pass / previous chunk (HBM-read-bound) on a side stream that forks
 * from and joins `stream` (CUDA-graph capturable).  `fine` may be NULL (N_importance == 0). */
typedef struct {
  const float* z_vals;      /* [N,S] */
  const float* noise;       /* [N,S] or NULL */
  int S;
  const NerfNetParams* net;
  const void* packed;
  const float* raw;         /* [N,S,4] of the training-mode pass */
  const NerfTrainSave* save;
  const float* g_rgb;       /* dL/drgb_map [N,3] */
  const NerfNetGrads* grads;
} NerfBwdPass;
int nerf_b200_render_rays_bwd_tc(const float* rays, int64_t N, const NerfRenderCfg* cfg, const NerfBwdPass* coarse,
                                 const NerfBwdPass* fine, void* workspace, size_t workspace_bytes, void* stream);
size_t nerf_b200_render_rays_bwd_tc_workspace_bytes(int64_t N, int S_coarse, const NerfNetParams* net_coarse, int S_fine,
                                                    const NerfNetParams* net_fine);
/* exact mode (csrc/bwd_simt.cuh): fp32 recompute with saved activations + fp32 CUDA-core GEMMs; any network
 * the exact forward supports (with or without view directions). */
int nerf_b200_march_bwd(const float* rays, const float* z_vals, const float* noise, int64_t N, int S,
                        const NerfNetParams* net, const void* packed, const NerfRenderCfg* cfg,
                        const float* g_rgb, const NerfNetGrads* grads, void* workspace,
                        size_t workspace_bytes, void* stream);
size_t nerf_b200_march_bwd_workspace_bytes(int64_t N, int S, const NerfNetParams* net);

/* ---- the two ends of the optimisation step (SURVEY 8f rank 2; csrc/train_step.cuh) ------------------------------
 *      mse_seed : img2mse (run_nerf_helpers.py:9; run_nerf.py:764-772): *loss_accum += mean((rgb - target)^2) and
 *                 g_rgb = 2 (rgb - target) / (3 N) * grad_scale  (grad_scale = 1 / world_size under data parallelism)
 *      adam_step: torch.optim.Adam(betas, eps) (run_nerf.py:207, :776) over one flat fp32 parameter buffer, with the
 *                 reference's learning-rate decay (run_nerf.py:778-783) evaluated on the device; state = float[4]:
 *                 [1] = steps taken so far, [2] = rate of the last step.  grads are multiplied by grad_mul first. ---- */
int nerf_b200_mse_seed(const float* rgb, const float* target, int64_t N, float grad_scale, float* g_rgb, float* loss_accum, void* stream);
int nerf_b200_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n, float* state,
                        float lr0, float decay_rate, float decay_steps, float beta1, float beta2, float eps, float grad_mul, void* stream);

/* ---- device-time accounting of the dominant kernels (march_tc2 / dgrad_tc2 / wgrad_tc) for bench.py's roofline:
 *      when enabled, every launch is bracketed by CUDA events on its own stream; read() synchronises
 *      those events, returns the summed kernel time [ms], the launch count and the algorithmic
 *      FLOPs those launches performed (SURVEY 8d: 2 x MACs of the reference layers x rows), and
 *      resets the accumulators. ------------------------------------------------------------------- */
int nerf_b200_timing_enable(int on);
int nerf_b200_timing_read(double* kernel_ms, int64_t* launches, double* algorithmic_flops);
/* same, also split by kind: kind_ms[0] forward passes, [1] dgrad chains, [2] weight-gradient kernels */
int nerf_b200_timing_read_kinds(double* kernel_ms, int64_t* launches, double* algorithmic_flops, double* kind_ms);

/* ---- number of kernels launched by this library since load (bench.py's gpu_launches) ---------- */
int64_t nerf_b200_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* NERF_B200_H_ */
