"""Golden fixtures of the UNMODIFIED reference that the tests used to take from a live copy of it.

    python oracle/gen_reference_runs.py keras [out_dir]      # CPU
    python oracle/gen_reference_runs.py gpu [out_dir]        # needs CUDA; the reference's own GPU runs

The reference is found through oracle/ref_import.py ($NERF_REFERENCE, else the copy oracle/fetch_reference.py leaves in
oracle/_ref/, which is copied along with the repository).  out_dir defaults to tests/golden/.  Writes

  keras_weights.npz   NeRF.load_weights_from_keras of the reference (run_nerf_helpers.py:121-148) on the seeded Keras-style
                      weight list of tests/test_host_cpu.py: the state_dict keys in order, their shapes and a seeded sample
  reference_gpu_trained_lego_1024.npz
                      the reference's render() on cuda:0 of the 1024 rays of trained_lego_1024.npz with the trained networks,
                      fp32 and TF32 matmuls (TF32 is the default of the reference's pinned torch 1.11)
  dropin_train.npz    the reference's own train() (run_nerf.py:701-873) for K_ITERS iterations on a small synthetic
                      blender-format dataset, started from the seeded synth.nerf_state(0) / (1) weights: each iteration's ray
                      batch, target and CUDA generator state before render(), every img2mse value and a seeded sample of the
                      parameter update; then, from the starting weights again, a sample of the gradients of one more step on
                      recorded rays (perturb = 0) and a 40x40 render(c2w=...) under no_grad.  tests/test_gpu_dropin.py replays it
                      through nerf_pytorch_b200.dropin.
"""
import argparse
import json
import os
import sys
import tempfile
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_import, synth  # noqa: E402

K_ITERS = 6
N_RAND = 512
SAMPLE = 512                      # sampled entries per parameter tensor (all of the smaller ones)
NET_KEYS = ("network_fn", "network_fine")
TRAIN_ARGV = ["--dataset_type", "blender", "--N_rand", str(N_RAND), "--N_samples", "64", "--N_importance", "128", "--use_viewdirs",
              "--white_bkgd", "--lrate_decay", "500", "--raw_noise_std", "0"]


def keras_weight_list():
    """the Keras-style weight list (kernel [in, out], bias [out] per layer) of tests/test_host_cpu.py"""
    rng = np.random.default_rng(0)
    shapes = [(63, 256)] + [(256, 256)] * 4 + [(319, 256)] + [(256, 256)] * 2 + [(256, 256), (283, 128), (128, 3), (256, 1)]
    weights = []
    for (i, o) in shapes:
        weights += [rng.standard_normal((i, o)).astype(np.float32), rng.standard_normal((o,)).astype(np.float32)]
    return weights


def sample_index(rng, n):
    return np.arange(n, dtype=np.int64) if n <= SAMPLE else np.sort(rng.choice(n, SAMPLE, replace=False)).astype(np.int64)


def gen_keras(out):
    _, rh = ref_import.load()
    r = rh.NeRF(D=8, W=256, input_ch=63, input_ch_views=27, output_ch=5, skips=[4], use_viewdirs=True)
    r.load_weights_from_keras(keras_weight_list())
    rng = np.random.default_rng(1)
    sd = r.state_dict()
    fx = {"keys": np.array(list(sd.keys()))}
    for k, v in sd.items():
        flat = v.detach().numpy().reshape(-1)
        idx = sample_index(rng, flat.size)
        fx[f"{k}__shape"] = np.array(v.shape, np.int64)
        fx[f"{k}__idx"], fx[f"{k}__val"] = idx, flat[idx]
    np.savez_compressed(os.path.join(out, "keras_weights.npz"), **fx)


def write_dataset(base, n=(8, 2, 2), H=40):
    """a small blender-format dataset (transforms_*.json + RGBA PNGs of a coloured disc) on the lego orbit"""
    import cv2
    ang = 0.6911112070083618
    rng = np.random.default_rng(0)
    yy, xx = np.mgrid[0:H, 0:H].astype(np.float32) / H
    k = 0
    for split, cnt in zip(("train", "val", "test"), n):
        os.makedirs(os.path.join(base, split), exist_ok=True)
        frames = []
        for i in range(cnt):
            th, ph = 360.0 * k / sum(n), -30.0 + 10.0 * (k % 3)
            c, s = np.cos(np.radians(th)), np.sin(np.radians(th))
            cp, sp = np.cos(np.radians(ph)), np.sin(np.radians(ph))
            t = np.array([[1, 0, 0, 0], [0, 1, 0, 0], [0, 0, 1, 4.0], [0, 0, 0, 1]], np.float64)
            rp = np.array([[1, 0, 0, 0], [0, cp, -sp, 0], [0, sp, cp, 0], [0, 0, 0, 1]], np.float64)
            rt = np.array([[c, 0, -s, 0], [0, 1, 0, 0], [s, 0, c, 0], [0, 0, 0, 1]], np.float64)
            c2w = np.array([[-1, 0, 0, 0], [0, 0, 1, 0], [0, 1, 0, 0], [0, 0, 0, 1]], np.float64) @ rt @ rp @ t
            disc = ((xx - 0.5) ** 2 + (yy - 0.5) ** 2) < 0.12
            img = np.zeros((H, H, 4), np.float32)
            img[..., 0] = 0.5 + 0.5 * np.sin(6 * xx + th / 40.0)
            img[..., 1] = 0.5 + 0.5 * np.cos(5 * yy + 0.3 * k)
            img[..., 2] = 0.3 + 0.4 * xx * yy + 0.2 * rng.random()
            img[..., 3] = disc
            img[..., :3] *= disc[..., None]
            png = (np.clip(img[..., [2, 1, 0, 3]], 0, 1) * 255).astype(np.uint8)          # cv2 writes BGRA
            cv2.imwrite(os.path.join(base, split, f"r_{i}.png"), png)
            frames.append({"file_path": f"./{split}/r_{i}", "transform_matrix": c2w.tolist()})
            k += 1
        with open(os.path.join(base, f"transforms_{split}.json"), "w") as f:
            json.dump({"camera_angle_x": ang, "frames": frames}, f)


def stand_ins():
    """cv2-backed imageio and argparse-backed configargparse (neither package is installed), empty matplotlib"""
    import cv2
    imageio = types.ModuleType("imageio")
    imageio.imread = lambda f, *a, **k: cv2.imread(f, cv2.IMREAD_UNCHANGED)[..., [2, 1, 0, 3]]
    imageio.imwrite = lambda f, im, *a, **k: cv2.imwrite(f, np.asarray(im)[..., ::-1])
    imageio.mimwrite = lambda *a, **k: None
    cfg = types.ModuleType("configargparse")

    class ArgumentParser(argparse.ArgumentParser):
        def add_argument(self, *a, **k):
            k.pop("is_config_file", None)
            return super().add_argument(*a, **k)
    cfg.ArgumentParser = ArgumentParser
    mpl, plt = types.ModuleType("matplotlib"), types.ModuleType("matplotlib.pyplot")
    mpl.pyplot = plt
    for name, mod in (("imageio", imageio), ("configargparse", cfg), ("matplotlib", mpl), ("matplotlib.pyplot", plt)):
        sys.modules.setdefault(name, mod)


def to_np(t):
    return t.detach().float().cpu().numpy()


def gen_tf32(rn, out):
    """the reference's render() of trained_lego_1024's rays on cuda:0, fp32 and TF32"""
    w = np.load(os.path.join(ROOT, "tests", "golden", "trained_weights.npz"))
    fx = np.load(os.path.join(ROOT, "tests", "golden", "trained_lego_1024.npz"))
    sb = synth.ray_batch("lego", int(fx["N"]), seed=int(fx["ray_seed"]))
    res = {"N": fx["N"], "ray_seed": fx["ray_seed"]}
    for tag, tf32 in (("fp32", False), ("tf32", True)):
        torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = tf32
        with tempfile.TemporaryDirectory() as tmp:
            os.makedirs(os.path.join(tmp, "e"))
            args = argparse.Namespace(multires=10, multires_views=4, i_embed=0, use_viewdirs=True, N_importance=128, N_samples=64, netdepth=8,
                                      netwidth=256, netdepth_fine=8, netwidth_fine=256, netchunk=65536, lrate=5e-4, basedir=tmp, expname="e",
                                      ft_path=None, no_reload=True, perturb=0.0, white_bkgd=True, raw_noise_std=0.0, dataset_type="blender",
                                      no_ndc=False, lindisp=False)
            _, te, _, _, _ = rn.create_nerf(args)
        for t, key in (("c", "network_fn"), ("f", "network_fine")):
            te[key].load_state_dict({k[2:]: torch.from_numpy(w[k]).cuda() for k in w.files if k.startswith(t + ".")})
        te.update(near=2., far=6.)
        with torch.no_grad():
            rgb, disp, acc, ex = rn.render(sb["H"], sb["W"], sb["K"], chunk=32768, rays=torch.from_numpy(sb["rays"]).cuda(), **te)
        res.update({f"{tag}_rgb_map": to_np(rgb), f"{tag}_acc_map": to_np(acc), f"{tag}_rgb0": to_np(ex["rgb0"]), f"{tag}_acc0": to_np(ex["acc0"])})
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    np.savez_compressed(os.path.join(out, "reference_gpu_trained_lego_1024.npz"), **res)


def gen_dropin(rn, out):
    """the reference's train() for K_ITERS iterations, recorded for a replay through the drop-in"""
    init = [synth.nerf_state(0), synth.nerf_state(1)]
    rec = {"rays": [], "rng": [], "mse_x": [], "mse_y": [], "loss": []}
    captured = {}
    orig_create, orig_render, orig_mse = rn.create_nerf, rn.render, rn.img2mse

    def spy_create(args):
        res = orig_create(args)
        for key, sd in zip(NET_KEYS, init):
            res[0][key].load_state_dict({k: torch.from_numpy(v).cuda() for k, v in sd.items()})
        captured["res"], captured["args"] = res, args
        return res

    def spy_render(H, W, K, rays=None, **kw):
        rec["rays"].append(to_np(rays))
        rec["rng"].append(torch.cuda.get_rng_state().numpy().copy())
        return orig_render(H, W, K, rays=rays, **kw)

    def spy_mse(x, y):
        v = orig_mse(x, y)
        rec["mse_y"].append(to_np(y))
        rec["loss"].append(float(v))
        return v

    with tempfile.TemporaryDirectory() as tmp:
        data = os.path.join(tmp, "data")
        write_dataset(data)
        rn.create_nerf, rn.render, rn.img2mse = spy_create, spy_render, spy_mse
        rn.trange = lambda a, b: range(a, a + K_ITERS)            # N_iters = 200001 is hard-coded (run_nerf.py:701)
        old_argv = sys.argv
        sys.argv = ["run_nerf.py", "--datadir", data, "--basedir", os.path.join(tmp, "logs"), "--expname", "ref"] + TRAIN_ARGV
        np.random.seed(0)
        torch.manual_seed(0)
        try:
            rn.train()
        finally:
            sys.argv = old_argv
            rn.create_nerf, rn.render, rn.img2mse = orig_create, orig_render, orig_mse
        torch.cuda.synchronize()
        with open(os.path.join(data, "transforms_test.json")) as f:
            c2w = np.array(json.load(f)["frames"][0]["transform_matrix"], np.float32)[:3, :4]
        with open(os.path.join(data, "transforms_train.json")) as f:
            pose = np.array(json.load(f)["frames"][1]["transform_matrix"], np.float32)[:3, :4]
    assert len(rec["rays"]) == K_ITERS and len(rec["loss"]) == 2 * K_ITERS
    tr, te = captured["res"][0], captured["res"][1]
    args = {k: v for k, v in vars(captured["args"]).items() if k not in ("datadir", "basedir", "expname", "config")}
    rng = np.random.default_rng(2)
    fx = {"args": np.array(json.dumps(args)), "rays": np.stack(rec["rays"]), "target": np.stack(rec["mse_y"][0::2]),
          "rng_state": np.stack(rec["rng"]), "loss": np.array(rec["loss"], np.float64), "c2w": c2w}
    # parameter update after K_ITERS steps, sampled
    for key, sd0 in zip(NET_KEYS, init):
        for k, v in tr[key].state_dict().items():
            upd = (to_np(v).astype(np.float64) - sd0[k].astype(np.float64)).reshape(-1)
            idx = sample_index(rng, upd.size)
            fx[f"upd.{key}.{k}.idx"], fx[f"upd.{key}.{k}.val"] = idx, upd[idx]
    # from the starting weights again: gradients of one more training-mode step (perturb = 0) on a recorded-here batch
    H0 = W0 = 40
    f0 = 0.5 * W0 / np.tan(0.5 * 0.6911112070083618)
    K0 = np.array([[f0, 0, 0.5 * W0], [0, f0, 0.5 * H0], [0, 0, 1]])
    for key, sd in zip(NET_KEYS, init):
        tr[key].load_state_dict({k: torch.from_numpy(v).cuda() for k, v in sd.items()})
    ro, rd = rn.get_rays(H0, W0, K0, torch.from_numpy(pose).cuda())
    sel = torch.randperm(H0 * W0)[:N_RAND]
    batch_rays = torch.stack([ro.reshape(-1, 3)[sel], rd.reshape(-1, 3)[sel]], 0)
    tgt = torch.rand(N_RAND, 3)
    kw = dict(tr); kw.update(near=2., far=6., perturb=0.)
    for key in NET_KEYS:
        for p in kw[key].parameters():
            p.grad = None
    rgb, _, _, extras = rn.render(H0, W0, K0, chunk=32768, rays=batch_rays, verbose=False, retraw=True, **kw)
    (rn.img2mse(rgb, tgt) + rn.img2mse(extras["rgb0"], tgt)).backward()
    fx["grad_rays"], fx["grad_target"] = to_np(batch_rays), to_np(tgt)
    for key in NET_KEYS:
        for k, p in kw[key].named_parameters():
            g = to_np(p.grad).astype(np.float64).reshape(-1)
            idx = sample_index(rng, g.size)
            fx[f"grad.{key}.{k}.idx"], fx[f"grad.{key}.{k}.val"] = idx, g[idx]
    # same starting weights -> image through render(c2w=...) under no_grad (run_nerf.py:154 call shape)
    kw_t = dict(te); kw_t.update(near=2., far=6.)
    with torch.no_grad():
        img = rn.render(H0, W0, K0, chunk=32768, c2w=torch.from_numpy(c2w).cuda(), **kw_t)
    fx["render_rgb"], fx["render_acc"], fx["render_rgb0"] = to_np(img[0]), to_np(img[2]), to_np(img[3]["rgb0"])
    np.savez_compressed(os.path.join(out, "dropin_train.npz"), **fx)
    print("dropin_train: losses", rec["loss"])


def main():
    mode = sys.argv[1]
    out = sys.argv[2] if len(sys.argv) > 2 else os.path.join(ROOT, "tests", "golden")
    os.makedirs(out, exist_ok=True)
    assert ref_import.available(), f"reference not found at {ref_import.REF} (oracle/fetch_reference.py)"
    if mode == "keras":
        gen_keras(out)
        return
    assert mode == "gpu" and torch.cuda.is_available(), "usage: gen_reference_runs.py keras|gpu [out_dir] (gpu needs CUDA)"
    stand_ins()
    rn, _ = ref_import.load()
    torch.set_default_tensor_type("torch.cuda.FloatTensor")            # what run_nerf.py:876 does under __main__
    gen_tf32(rn, out)
    gen_dropin(rn, out)
    print("done")


if __name__ == "__main__":
    main()
