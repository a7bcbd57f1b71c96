"""The drop-in against the reference's own training run: the unmodified reference script's `train()` ran K iterations on a
small synthetic blender-format dataset (oracle/gen_reference_runs.py: argument parsing, data loading, ray batching,
`create_nerf` (run_nerf.py:640), `render(..., retraw=True)` (:760), the two MSE terms, `loss.backward()`,
`optimizer.step()` and the learning-rate decay (:764-784)), and tests/golden/dropin_train.npz holds what it saw and did:
each iteration's ray batch, target and CUDA generator state before `render()`, every loss term and a seeded sample of
the parameter update.  Here the names `nerf_pytorch_b200.dropin.patch` rebinds on a module run the same iterations from
the same starting weights with the same arguments.

Checks: same loss trajectory, same parameter update after K steps (within the tensor-core budget), same gradients of one
more step from identical weights and rays, same rendered image from the same weights through `render(c2w=...)` under
no_grad.  The measured values are also written to parity_dropin.json, next to the other parity records."""
import argparse
import json
import os
import types

import numpy as np
import pytest
import torch

from conftest import ROOT, rel_l2

pytestmark = pytest.mark.gpu
NET_KEYS = ("network_fn", "network_fine")


def _sampled(fx, kind, tensors):
    """{name: (ours at the stored indices, reference's stored values)} for every parameter tensor"""
    out = {}
    for key in NET_KEYS:
        for k, t in tensors(key):
            idx = fx[f"{kind}.{key}.{k}.idx"]
            out[f"{key}.{k}"] = (t.detach().double().reshape(-1).cpu().numpy()[idx], fx[f"{kind}.{key}.{k}.val"])
    return out


def test_reference_train_runs_unchanged_through_the_dropin(tmp_path, golden):
    import nerf_pytorch_b200 as nb
    from nerf_pytorch_b200 import dropin
    from oracle import synth
    fx = golden("dropin_train")
    K_ITERS = fx["rays"].shape[0]
    args = argparse.Namespace(**json.loads(str(fx["args"])), basedir=str(tmp_path), expname="patched")
    os.makedirs(tmp_path / "patched")
    init = [synth.nerf_state(0), synth.nerf_state(1)]
    torch.set_default_tensor_type("torch.cuda.FloatTensor")            # what run_nerf.py:876 does under __main__
    try:
        launches0 = nb.launch_count()
        pat = dropin.patch(types.ModuleType("run_nerf"), set_default_device=False)
        tr, te, start, grad_vars, optimizer = pat.create_nerf(args)
        assert isinstance(tr["network_fn"], nb.NeRF) and start == 0
        for key, sd in zip(NET_KEYS, init):
            tr[key].load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
        for kw in (tr, te):
            kw.update(near=2., far=6.)                                  # blender bounds (run_nerf.py:573-574)
        H = W = 40
        focal = 0.5 * W / np.tan(0.5 * 0.6911112070083618)
        K = np.array([[focal, 0, 0.5 * W], [0, focal, 0.5 * H], [0, 0, 1]])
        # the reference's loop body (run_nerf.py:760-784) on the batches its train() drew, from its generator states
        losses = []
        for i in range(K_ITERS):
            torch.cuda.set_rng_state(torch.from_numpy(fx["rng_state"][i]))
            target = torch.from_numpy(fx["target"][i]).cuda()
            rgb, disp, acc, extras = pat.render(H, W, K, chunk=args.chunk, rays=torch.from_numpy(fx["rays"][i]).cuda(), verbose=i < 10,
                                                retraw=True, **tr)
            optimizer.zero_grad()
            terms = [nb.img2mse(rgb, target), nb.img2mse(extras["rgb0"], target)]
            losses += [float(t) for t in terms]
            (terms[0] + terms[1]).backward()
            optimizer.step()
            for g in optimizer.param_groups:                            # global_step = start + i (run_nerf.py:779-783, :873)
                g["lr"] = args.lrate * 0.1 ** ((start + i) / (args.lrate_decay * 1000))
        torch.cuda.synchronize()
        assert nb.launch_count() > launches0
        loss_r = fx["loss"]
        assert len(losses) == len(loss_r) == 2 * K_ITERS                # img2mse is called twice per iteration (:764, :771)
        stats = {"loss_reference": loss_r.tolist(), "loss_patched": losses}
        stats["loss_max_rel_dev"] = float(np.max(np.abs(np.array(losses) - loss_r) / loss_r))
        # parameter update after K iterations (Adam, same lr schedule), on the stored sample of every tensor
        upd = {}
        init_t = {key: {k: torch.from_numpy(v).cuda() for k, v in sd.items()} for key, sd in zip(NET_KEYS, init)}
        for name, (dp, dr) in _sampled(fx, "upd", lambda key: [(k, v - init_t[key][k]) for k, v in tr[key].state_dict().items()]).items():
            upd[name] = {"rel": rel_l2(dp, dr), "cos": float(dp @ dr / (np.linalg.norm(dp) * np.linalg.norm(dr) + 1e-30))}
        stats["update"] = upd
        stats["update_cos_min"] = min(v["cos"] for v in upd.values())
        stats["update_rel_median"] = float(np.median([v["rel"] for v in upd.values()]))
        # gradients of one more reference-style step from IDENTICAL weights and rays (perturb = 0):
        # Adam's first steps move every element by ~lr * sign(g), so elements whose gradient is noise-level make the
        # UPDATE vectors of some tensors decorrelate (recorded above) even when the gradients agree; the gate is on the gradients
        for key, sd in zip(NET_KEYS, init):
            tr[key].load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
        kw = dict(tr); kw.update(perturb=0.)
        for key in NET_KEYS:
            for p_ in kw[key].parameters():
                p_.grad = None
        tgt = torch.from_numpy(fx["grad_target"]).cuda()
        rgb, disp, acc, extras = pat.render(H, W, K, chunk=32768, rays=torch.from_numpy(fx["grad_rays"]).cuda(), verbose=False, retraw=True, **kw)
        (nb.img2mse(rgb, tgt) + nb.img2mse(extras["rgb0"], tgt)).backward()
        grads = _sampled(fx, "grad", lambda key: [(k, p_.grad) for k, p_ in kw[key].named_parameters()])
        gstats = {name: rel_l2(gp, gr) for name, (gp, gr) in grads.items()}
        stats["grad_rel"] = gstats
        stats["grad_rel_median"] = float(np.median(list(gstats.values())))
        stats["grad_rel_max"] = float(max(gstats.values()))
        allp = np.concatenate([gp for gp, _ in grads.values()])
        allr = np.concatenate([gr for _, gr in grads.values()])
        stats["grad_cos_all"] = float(allr @ allp / (np.linalg.norm(allr) * np.linalg.norm(allp)))
        # same weights -> same image through render(c2w=...) under no_grad (run_nerf.py:154 call shape)
        with torch.no_grad():
            img_p = pat.render(H, W, K, chunk=32768, c2w=torch.from_numpy(fx["c2w"]).cuda(), **te)
        stats["render_rgb_rel"] = rel_l2(img_p[0].cpu().numpy(), fx["render_rgb"])
        stats["render_acc_rel"] = rel_l2(img_p[2].cpu().numpy(), fx["render_acc"])
        stats["render_rgb0_rel"] = rel_l2(img_p[3]["rgb0"].cpu().numpy(), fx["render_rgb0"])
        os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
        with open(os.path.join(ROOT, "gpurun_out", "parity_dropin.json"), "w") as f:
            json.dump(stats, f, indent=1)
        print({k: v for k, v in stats.items() if k not in ("update", "grad_rel")})
        assert stats["render_rgb_rel"] < 1e-3 and stats["render_acc_rel"] < 1e-3, stats
        assert stats["loss_max_rel_dev"] < 1e-3, stats
        assert stats["grad_rel_median"] < 3e-2 and stats["grad_rel_max"] < 1.5e-1 and stats["grad_cos_all"] > 0.999, {k: v for k, v in stats.items() if k != "update"}
        assert stats["update_rel_median"] < 0.1, stats["update_rel_median"]
    finally:
        torch.set_default_tensor_type("torch.FloatTensor")
