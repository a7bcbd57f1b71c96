"""Discriminating parity: fixtures WITH STRUCTURE (oracle/gen_trained.py: networks trained by the unmodified reference for
a few hundred CPU steps on an analytic scene, so acc spans 0..1 and the weights are peaked) at 1024 rays, BASELINE config 3's
shape (4096 fern NDC rays), the fused path's `weights` (coarse and fine) and sorted z, and the gradients on the trained
networks.  Every measured deviation is written to gpurun_out/parity_r02.json (committed as profiles/parity_r02.json)."""
import ctypes as C
import json
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, ROOT, load_golden, rel_l2

pytestmark = pytest.mark.gpu
needs_trained = pytest.mark.skipif(not os.path.isfile(os.path.join(GOLDEN, "trained_weights.npz")), reason="tests/golden/trained_weights.npz missing (oracle/gen_trained.py)")


@pytest.fixture(scope="module")
def G():
    import gpu_common
    return gpu_common


def _record(name, value):
    path = os.path.join(ROOT, "gpurun_out", "parity_r02.json")
    os.makedirs(os.path.dirname(path), exist_ok=True)
    data = {}
    if os.path.isfile(path):
        with open(path) as f:
            data = json.load(f)
    data[name] = value
    with open(path, "w") as f:
        json.dump(data, f, indent=1, sort_keys=True)


def _trained_nets(G):
    w = load_golden("trained_weights")
    nets = []
    for tag in ("c", "f"):
        nets.append(G.make_net({k[2:]: v for k, v in w.items() if k.startswith(tag + ".")}))
    return nets


def _fwd_with_weights(G, nets, packed, Sc, Ni, white, prec):
    """nerf_b200_render_rays_fwd through the C ABI with the weights of BOTH passes requested"""
    lib = G._lib.load()
    N = packed.shape[0]
    Sf = Sc + Ni
    cfg = G._lib.NerfRenderCfg()
    cfg.N_samples, cfg.N_importance, cfg.multires, cfg.multires_views = Sc, Ni, 10, 4
    cfg.lindisp, cfg.perturb, cfg.white_bkgd, cfg.ray_stride = 0, 0, int(white), 11
    cfg.precision = G._lib.PREC_TC_FP16 if prec == "tc_fp16" else G._lib.PREC_FP32
    z = lambda *s: torch.zeros(s, device=G.DEV)
    o = dict(rgb0=z(N, 3), disp0=z(N), acc0=z(N), w0=z(N, Sc), raw0=z(N, Sc, 4), rgb=z(N, 3), disp=z(N), acc=z(N), w=z(N, Sf), raw=z(N, Sf, 4),
             z_c=z(N, Sc), z_f=z(N, Sf), z_std=z(N))
    out_c = G._lib.NerfPassOut(G.ptr(o["rgb0"]), G.ptr(o["disp0"]), G.ptr(o["acc0"]), C.c_void_p(0), G.ptr(o["w0"]), G.ptr(o["raw0"]))
    out_f = G._lib.NerfPassOut(G.ptr(o["rgb"]), G.ptr(o["disp"]), G.ptr(o["acc"]), C.c_void_p(0), G.ptr(o["w"]), G.ptr(o["raw"]))
    pc, pf = nets[0].net_params(), nets[1].net_params()
    tc = prec == "tc_fp16"
    t_vals, u_det = torch.linspace(0., 1., Sc, device=G.DEV), torch.linspace(0., 1., Ni, device=G.DEV)
    ws_bytes = lib.nerf_b200_march_workspace_bytes(N, Sf)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=G.DEV)
    rays = G.dev(packed)
    G._lib.check(lib.nerf_b200_render_rays_fwd(G.ptr(rays), N, C.byref(cfg), C.byref(pc), G.ptr(nets[0].packed() if tc else None), C.byref(pf),
                                               G.ptr(nets[1].packed() if tc else None), G.ptr(t_vals), G.ptr(u_det), None, None, None, None,
                                               G.ptr(o["z_c"]), C.byref(out_c), G.ptr(o["z_f"]), G.ptr(o["z_std"]), C.byref(out_f), G.ptr(ws), ws_bytes,
                                               G.stream()), "render_rays_fwd")
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in o.items()}


def _finite_rel(a, b):
    m = np.isfinite(a) & np.isfinite(b)
    return rel_l2(a[m], b[m]), bool(np.array_equal(np.isnan(a), np.isnan(b)))


@needs_trained
@pytest.mark.parametrize("prec", ["fp32", "tc_fp16"])
def test_trained_networks_1024_rays_outputs_weights_and_z(G, prec):
    fx = load_golden("trained_lego_1024")
    sb = G.synth.ray_batch("lego", int(fx["N"]), seed=int(fx["ray_seed"]))
    packed = G.O.pack_rays(sb["H"], sb["W"], sb["K"], sb["rays"][0], sb["rays"][1], False, 2.0, 6.0, True).astype(np.float32)
    nets = _trained_nets(G)
    o = _fwd_with_weights(G, nets, packed, 64, 128, True, prec)
    st = {"acc_min": float(fx["acc_map"].min()), "acc_max": float(fx["acc_map"].max()), "rgb_std": float(fx["rgb_map"].std())}
    for k, ref in (("rgb", "rgb_map"), ("acc", "acc_map"), ("rgb0", "rgb0"), ("acc0", "acc0"), ("w0", "w_coarse"), ("w", "w_fine"), ("z_f", "z_fine"),
                   ("z_std", "z_std")):
        st[ref] = rel_l2(o[k], fx[ref])
    for k, ref in (("raw0", "raw_coarse"), ("raw", "raw_fine")):            # stored for the first 256 rays only
        st[ref] = rel_l2(o[k][:256], fx[ref])
    st["disp_map"], st["disp_nan_mask_equal"] = _finite_rel(o["disp"], fx["disp_map"])
    st["disp0"], st["disp0_nan_mask_equal"] = _finite_rel(o["disp0"], fx["disp0"])
    _record(f"trained_lego_1024_{prec}", st)
    print(prec, {k: (float("%.3g" % v) if isinstance(v, float) else v) for k, v in st.items()})
    st["disp_nan_mask_mismatch"] = float(np.mean(np.isnan(o["disp"]) != np.isnan(fx["disp_map"])))
    _record(f"trained_lego_1024_{prec}", st)
    assert st["acc_max"] - st["acc_min"] > 0.5                      # the fixture has structure
    _check_trained_gates(st, prec)


def _check_trained_gates(st, prec):
    """Gates on networks WITH structure (measured values: profiles/parity_r02.json).

    fp32 (exact mode): the coarse pass agrees to fp32 round-off (<= 2e-5); the fine pass additionally sees the resampling's
    sensitivity -- a 1e-7 difference in a coarse weight can move an inverse-CDF sample across a bin knot (SURVEY App. D quirk 5),
    the sample lands elsewhere on the ray and the fine maps move by ~1e-4 (the reference itself shows this between BLAS builds).
    tc_fp16: 11-bit operands.  Coarse maps <= 2e-4; the fine maps inherit knot flips from 5e-4-level coarse weight deviations and
    their own operand rounding: rgb_map <= 3e-3 (measured 0.5-1.8e-3).  The north star's 1e-4 is met on the default-initialised
    fixtures (tests/test_gpu_render.py) and by the coarse pass here, NOT by the fine pass of trained-like networks; the reference's
    own GPU default (TF32) deviates as much from its fp32 run (test_reference_tf32_deviates_as_much)."""
    if prec == "fp32":
        assert st["rgb0"] < 2e-5 and st["acc0"] < 2e-5, st
        assert st["rgb_map"] < 3e-4 and st["acc_map"] < 3e-4, st
        if "w_coarse" in st:
            assert st["w_coarse"] < 1e-5 and st["w_fine"] < 2e-3 and st["z_fine"] < 2e-3, st
        assert st["disp_nan_mask_mismatch"] == 0.0, st
    else:
        assert st["rgb0"] < 3e-4 and st["acc0"] < 3e-4, st
        assert st["rgb_map"] < 3e-3 and st["acc_map"] < 4e-3, st
        if "w_coarse" in st:
            assert st["w_coarse"] < 2e-3 and st["w_fine"] < 1e-1, st
        assert st["disp_nan_mask_mismatch"] < 0.02, st


@needs_trained
@pytest.mark.parametrize("prec", ["fp32", "tc_fp16"])
def test_config3_fern_ndc_4096_rays(G, prec):
    """BASELINE configs[2]: fern LLFF 504x378 NDC rays, N_rand = 4096, 64 + 128 samples, on the trained networks (the default
    initialisation gives acc0 == 0 on NDC rays: a vacuous coarse pass)."""
    fx = load_golden("fern_ndc_4096")
    sb = G.synth.ray_batch("fern", 4096, seed=int(fx["ray_seed"]))
    nets = _trained_nets(G)
    G.nb.set_precision(prec)
    try:
        with torch.no_grad():
            rgb, disp, acc, ex = G.nb.render(sb["H"], sb["W"], sb["K"], chunk=32768, rays=G.dev(sb["rays"]), ndc=True, near=0., far=1., use_viewdirs=True,
                                             network_fn=nets[0], network_fine=nets[1], network_query_fn=G.query_fn(), N_samples=64, N_importance=128,
                                             perturb=0., white_bkgd=False, raw_noise_std=0.)
    finally:
        G.nb.set_precision("tc_fp16")
    st = {"rgb_map": rel_l2(rgb.cpu().numpy(), fx["rgb_map"]), "acc_map": rel_l2(acc.cpu().numpy(), fx["acc_map"]),
          "rgb0": rel_l2(ex["rgb0"].cpu().numpy(), fx["rgb0"]), "acc0": rel_l2(ex["acc0"].cpu().numpy(), fx["acc0"]),
          "z_std": rel_l2(ex["z_std"].cpu().numpy(), fx["z_std"]), "acc_mean": float(fx["acc_map"].mean()), "acc0_mean": float(fx["acc0"].mean())}
    st["disp_map"], st["disp_nan_mask_equal"] = _finite_rel(disp.cpu().numpy(), fx["disp_map"])
    st["disp_nan_mask_mismatch"] = float(np.mean(np.isnan(disp.cpu().numpy()) != np.isnan(fx["disp_map"])))
    _record(f"fern_ndc_4096_{prec}", st)
    print(prec, st)
    assert st["acc0_mean"] > 0.1                                    # the coarse pass is not vacuous
    _check_trained_gates(st, prec)


@needs_trained
def test_psnr_on_the_analytic_scene_matches_the_reference(G):
    """PSNR of the trained networks against the analytic ground truth they were trained on (oracle/gen_trained.py: a shaded unit
    sphere on white) -- the reference's rendering (golden rgb_map) and ours must score the same (BASELINE config 5 asks for
    PSNR; no dataset exists in the container, so the scene is analytic)."""
    from oracle.gen_trained import sphere_targets
    fx = load_golden("trained_lego_1024")
    sb = G.synth.ray_batch("lego", int(fx["N"]), seed=int(fx["ray_seed"]))
    gt = sphere_targets(sb["rays"][0], sb["rays"][1])
    nets = _trained_nets(G)
    st = {"psnr_reference_fp32_cpu": float(-10.0 * np.log10(np.mean((fx["rgb_map"] - gt) ** 2)))}
    for prec in ("fp32", "tc_fp16"):
        G.nb.set_precision(prec)
        try:
            with torch.no_grad():
                rgb = G.nb.render(sb["H"], sb["W"], sb["K"], chunk=32768, rays=G.dev(sb["rays"]), ndc=False, near=2., far=6., use_viewdirs=True,
                                  network_fn=nets[0], network_fine=nets[1], network_query_fn=G.query_fn(), N_samples=64, N_importance=128,
                                  perturb=0., white_bkgd=True, raw_noise_std=0.)[0]
        finally:
            G.nb.set_precision("tc_fp16")
        st[f"psnr_{prec}"] = float(G.nb.mse2psnr(G.nb.img2mse(rgb, G.dev(gt))).item())
    _record("psnr_analytic_scene_trained_lego_1024", st)
    print(st)
    assert abs(st["psnr_fp32"] - st["psnr_reference_fp32_cpu"]) < 1e-3 and abs(st["psnr_tc_fp16"] - st["psnr_reference_fp32_cpu"]) < 2e-2, st


@needs_trained
def test_reference_tf32_deviates_as_much(G):
    """Context for the tensor-core gates: the UNMODIFIED reference on this GPU with TF32 matmuls (the default of its pinned torch
    1.11; same 10-bit mantissa as our fp16 operands) against its own fp32 run on the same GPU, next to our tc_fp16 path against
    that fp32 run -- on the trained networks, 1024 lego rays.  The reference's two GPU runs are stored in
    tests/golden/reference_gpu_trained_lego_1024.npz (oracle/gen_reference_runs.py)."""
    fx = load_golden("trained_lego_1024")
    sb = G.synth.ray_batch("lego", int(fx["N"]), seed=int(fx["ray_seed"]))
    rg = load_golden("reference_gpu_trained_lego_1024")
    assert int(rg["N"]) == int(fx["N"]) and int(rg["ray_seed"]) == int(fx["ray_seed"])
    r32 = {k: rg["fp32_" + k] for k in ("rgb_map", "acc_map", "rgb0", "acc0")}
    rtf = {k: rg["tf32_" + k] for k in ("rgb_map", "acc_map", "rgb0", "acc0")}
    nets = _trained_nets(G)
    with torch.no_grad():
        rgb, disp, acc, ex = G.nb.render(sb["H"], sb["W"], sb["K"], chunk=32768, rays=G.dev(sb["rays"]), ndc=False, near=2., far=6., use_viewdirs=True,
                                         network_fn=nets[0], network_fine=nets[1], network_query_fn=G.query_fn(), N_samples=64, N_importance=128,
                                         perturb=0., white_bkgd=True, raw_noise_std=0.)
    ours = {"rgb_map": rgb.cpu().numpy(), "acc_map": acc.cpu().numpy(), "rgb0": ex["rgb0"].cpu().numpy(), "acc0": ex["acc0"].cpu().numpy()}
    st = {}
    for k in ("rgb_map", "acc_map", "rgb0", "acc0"):
        st[k] = {"reference_gpu_fp32_vs_cpu_golden": rel_l2(r32[k], fx[k]), "reference_tf32_vs_reference_fp32": rel_l2(rtf[k], r32[k]),
                 "ours_tc_fp16_vs_reference_fp32": rel_l2(ours[k], r32[k])}
    _record("reference_tf32_context_trained_lego_1024", st)
    print(st)
    for k in ("rgb_map", "acc_map"):
        assert st[k]["ours_tc_fp16_vs_reference_fp32"] < 3.0 * max(st[k]["reference_tf32_vs_reference_fp32"], 3e-4), st


@needs_trained
@pytest.mark.parametrize("prec,backward", [("fp32", "exact"), ("tc_fp16", "exact"), ("tc_fp16", "tc")])
def test_trained_networks_gradients(G, prec, backward):
    fx = load_golden("trained_lego_grads")
    sb = G.synth.ray_batch("lego", int(fx["N"]), seed=int(fx["ray_seed"]))
    nets = _trained_nets(G)
    G.nb.set_precision(prec)
    G.nb.set_backward(backward)
    try:
        rgb, _, _, ex = G.nb.render(sb["H"], sb["W"], sb["K"], chunk=32768, rays=G.dev(sb["rays"]), ndc=False, near=2., far=6., use_viewdirs=True,
                                    network_fn=nets[0], network_fine=nets[1], network_query_fn=G.query_fn(), N_samples=64, N_importance=128,
                                    perturb=0., white_bkgd=True, raw_noise_std=0., retraw=True)
        target = G.dev(fx["target"])
        loss = G.nb.img2mse(rgb, target) + G.nb.img2mse(ex["rgb0"], target)
        loss.backward()
    finally:
        G.nb.set_precision("tc_fp16")
        G.nb.set_backward("tc")
    st = {"loss_rel": abs(float(loss) - float(fx["loss"])) / float(fx["loss"])}
    errs = {}
    for tag, net in (("c", nets[0]), ("f", nets[1])):
        for name, p in net.named_parameters():
            g = p.grad.detach().cpu().numpy().reshape(-1)
            idx, ref = fx[f"g_{tag}_{name}_idx"], fx[f"g_{tag}_{name}_val"]
            errs[f"{tag}.{name}"] = float(np.linalg.norm(g[idx] - ref) / max(np.linalg.norm(ref), 1e-12))
    st["per_tensor"] = errs
    st["median"], st["max"] = float(np.median(list(errs.values()))), float(max(errs.values()))
    _record(f"trained_grads_{prec}_{backward}", st)
    print(prec, backward, "median", st["median"], "max", st["max"], "loss_rel", st["loss_rel"])
    if prec == "fp32":
        assert st["median"] < 1e-3 and st["max"] < 2e-2, st
    else:
        assert st["median"] < 3e-2 and st["max"] < 2e-1, st
