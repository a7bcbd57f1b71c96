"""CPU-only checks: the C-ABI library builds, loads and exports every symbol include/nerf_b200.h
declares; the Python host mirrors the reference's interface (names, signatures, state_dict keys,
kwargs dict) and refuses to run without CUDA instead of falling back."""
import ctypes
import inspect
import os
import re
import types

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def nb():
    import __graft_entry__ as ge
    ge.build()
    import nerf_pytorch_b200
    return nerf_pytorch_b200


def test_library_exports_every_declared_symbol(nb):
    hdr = open(os.path.join(ROOT, "include", "nerf_b200.h")).read()
    declared = set(re.findall(r"\b(nerf_b200_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 20
    lib = ctypes.CDLL(os.path.join(ROOT, "nerf-pytorch_b200", "libnerf_b200.so"))
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in the header but not exported"
    from nerf_pytorch_b200 import _lib
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    assert _lib.load().nerf_b200_abi_version() == 1


def test_struct_layout_matches_header(nb):
    from nerf_pytorch_b200 import _lib
    assert ctypes.sizeof(_lib.NerfNetParams) == 8 * 4 + (16 + 16 + 10) * 8
    assert ctypes.sizeof(_lib.NerfRenderCfg) == 12 * 4
    assert ctypes.sizeof(_lib.NerfPassOut) == 6 * 8
    assert ctypes.sizeof(_lib.NerfNetGrads) == (16 + 16 + 10) * 8


def test_interface_mirrors_reference_signatures(nb):
    """Same parameter names/defaults as run_nerf.py:69-72, :308-320, :262, run_nerf_helpers.py:196, :48, :68."""
    sig = lambda f: [(p.name, p.default) for p in inspect.signature(f).parameters.values()]
    assert sig(nb.render)[:11] == [("H", inspect._empty), ("W", inspect._empty), ("K", inspect._empty), ("chunk", 1024 * 32),
                                   ("rays", None), ("c2w", None), ("ndc", True), ("near", 0.), ("far", 1.),
                                   ("use_viewdirs", False), ("c2w_staticcam", None)]
    assert [n for n, _ in sig(nb.render_rays)] == ["ray_batch", "network_fn", "network_query_fn", "N_samples", "retraw", "lindisp",
                                                  "perturb", "N_importance", "network_fine", "white_bkgd", "raw_noise_std", "verbose", "pytest"]
    assert [n for n, _ in sig(nb.raw2outputs)] == ["raw", "z_vals", "rays_d", "raw_noise_std", "white_bkgd", "pytest"]
    assert [n for n, _ in sig(nb.sample_pdf)] == ["bins", "weights", "N_samples", "det", "pytest"]
    assert [n for n, _ in sig(nb.get_embedder)] == ["multires", "i"]
    assert [n for n, _ in sig(nb.NeRF.__init__)][1:] == ["D", "W", "input_ch", "input_ch_views", "output_ch", "skips", "use_viewdirs"]
    assert [n for n, _ in sig(nb.run_network)] == ["inputs", "viewdirs", "fn", "embed_fn", "embeddirs_fn", "netchunk"]


def test_state_dict_keys_are_the_reference_contract(nb):
    m = nb.NeRF(D=8, W=256, input_ch=63, input_ch_views=27, output_ch=5, skips=[4], use_viewdirs=True)
    from oracle import synth
    assert set(m.state_dict()) == set(synth.nerf_state(0))            # keys of run_nerf_helpers.py:79-94
    m.load_state_dict({k: torch.from_numpy(v) for k, v in synth.nerf_state(0).items()})
    assert m.pts_linears[5].weight.shape == (256, 319) and m.views_linears[0].weight.shape == (128, 283)
    assert sum(p.numel() for p in m.parameters()) == 595844           # SURVEY 0: params per network
    m2 = nb.NeRF(D=8, W=256, input_ch=63, input_ch_views=0, output_ch=4, skips=[4], use_viewdirs=False)
    assert "output_linear.weight" in m2.state_dict()


def test_nerf_forward_on_embedded_rows_matches_oracle(nb):
    from oracle import nerf_oracle as O, synth
    st = synth.nerf_state(3)
    m = nb.NeRF(D=8, W=256, input_ch=63, input_ch_views=27, output_ch=5, skips=[4], use_viewdirs=True)
    m.load_state_dict({k: torch.from_numpy(v) for k, v in st.items()})
    x = np.random.default_rng(0).standard_normal((33, 90)).astype(np.float32)
    with torch.no_grad():
        y = m(torch.from_numpy(x)).numpy()
    np.testing.assert_allclose(y, O.nerf_forward(st, x, 63, 27), rtol=2e-4, atol=2e-5)


def test_no_cpu_fallback(nb):
    m = nb.NeRF(D=8, W=256, input_ch=63, input_ch_views=27, output_ch=5, skips=[4], use_viewdirs=True)
    with pytest.raises(RuntimeError, match="CUDA"):
        nb.render_rays(torch.zeros(4, 11), m, None, 64)
    with pytest.raises(RuntimeError, match="CUDA"):
        nb.sample_pdf(torch.zeros(2, 8), torch.zeros(2, 7), 4, det=True)
    with pytest.raises(RuntimeError, match="CUDA"):
        nb.raw2outputs(torch.zeros(2, 4, 4), torch.zeros(2, 4), torch.zeros(2, 3))
    with pytest.raises(RuntimeError, match="CUDA"):
        nb.get_embedder(10, 0)[0](torch.zeros(3, 3))
    with pytest.raises(RuntimeError, match="CUDA"):
        m.packed()


def test_create_nerf_structure(nb, tmp_path):
    os.makedirs(tmp_path / "exp")
    args = types.SimpleNamespace(multires=10, multires_views=4, i_embed=0, use_viewdirs=True, N_importance=128, N_samples=64,
                                 netdepth=8, netwidth=256, netdepth_fine=8, netwidth_fine=256, netchunk=65536, lrate=5e-4,
                                 basedir=str(tmp_path), expname="exp", ft_path=None, no_reload=False, perturb=1.0,
                                 white_bkgd=True, raw_noise_std=0.0, dataset_type="blender", no_ndc=False, lindisp=False)
    tr, te, start, grad_vars, opt = nb.create_nerf(args, device="cpu")
    assert set(tr) == {"network_query_fn", "perturb", "N_importance", "network_fine", "N_samples", "network_fn", "use_viewdirs",
                       "white_bkgd", "raw_noise_std", "ndc", "lindisp"}                       # run_nerf.py:237-253
    assert te["perturb"] is False and te["raw_noise_std"] == 0.0 and start == 0               # :255-257
    assert len(grad_vars) == 48 and isinstance(opt, torch.optim.Adam)
    # checkpoint round trip in the reference's format (run_nerf.py:792-800, :215-233)
    torch.save({"global_step": 7, "network_fn_state_dict": tr["network_fn"].state_dict(),
                "network_fine_state_dict": tr["network_fine"].state_dict(), "optimizer_state_dict": opt.state_dict()},
               tmp_path / "exp" / "000007.tar")
    tr2, _, start2, _, _ = nb.create_nerf(args, device="cpu")
    assert start2 == 7
    assert torch.equal(tr2["network_fn"].pts_linears[0].weight, tr["network_fn"].pts_linears[0].weight)
    args.dataset_type = "llff"
    tr3 = nb.create_nerf(args, device="cpu")[0]
    assert "ndc" not in tr3 and "lindisp" not in tr3                                          # :250-253


def test_cached_parameter_list_follows_the_module(nb):
    """NeRF._named_params() (the cached list every render_rays call uses) equals named_parameters(), in its order, survives
    load_state_dict / deepcopy, and is rebuilt when a layer gets a NEW Parameter object."""
    import copy
    net = nb.NeRF(D=8, W=256, input_ch=63, input_ch_views=27, output_ch=5, skips=[4], use_viewdirs=True)
    def names_ids(n):
        return [(k, id(q)) for _, _, k, q in n._named_params()]
    ref = [(k, id(q)) for k, q in net.named_parameters()]
    assert names_ids(net) == ref and len(ref) == 24
    assert net._named_params() is net._named_params()                                   # cached
    net.load_state_dict(copy.deepcopy(net.state_dict()))
    assert names_ids(net) == ref                                                        # same Parameter objects
    twin = copy.deepcopy(net)
    assert names_ids(twin) == [(k, id(q)) for k, q in twin.named_parameters()]
    assert all(a[1] != b[1] for a, b in zip(names_ids(twin), ref))                      # the copy lists its own parameters
    net.rgb_linear.bias = torch.nn.Parameter(torch.zeros(3))
    assert names_ids(net) == [(k, id(q)) for k, q in net.named_parameters()] and names_ids(net) != ref
    plain = nb.NeRF(D=4, W=64, input_ch=63, input_ch_views=27, output_ch=4, skips=[], use_viewdirs=False)
    assert [k for _, _, k, _ in plain._named_params()] == [k for k, _ in plain.named_parameters()]


def test_keras_weight_import_matches_the_reference(nb, golden):
    """NeRF.load_weights_from_keras vs the reference's own (run_nerf_helpers.py:121-148) on a synthetic Keras-style weight list;
    the reference's state_dict (keys in order, shapes, a seeded sample of the entries) is tests/golden/keras_weights.npz."""
    from oracle.gen_reference_runs import keras_weight_list
    weights = keras_weight_list()
    m = nb.NeRF(D=8, W=256, input_ch=63, input_ch_views=27, output_ch=5, skips=[4], use_viewdirs=True)
    m.load_weights_from_keras(weights)
    assert torch.equal(m.pts_linears[5].weight, torch.from_numpy(weights[10].T)) and torch.equal(m.alpha_linear.bias, torch.from_numpy(weights[23]))
    ref = golden("keras_weights")
    sd = m.state_dict()
    assert list(sd.keys()) == [str(k) for k in ref["keys"]]
    for k, a in sd.items():
        assert list(a.shape) == ref[f"{k}__shape"].tolist(), k
        assert np.array_equal(a.numpy().reshape(-1)[ref[f"{k}__idx"]], ref[f"{k}__val"]), k


def test_dropin_patch_list_covers_the_seam(nb, monkeypatch):
    from nerf_pytorch_b200 import dropin
    for name in ("render", "render_rays", "batchify_rays", "raw2outputs", "create_nerf", "sample_pdf", "NeRF", "get_embedder"):
        assert name in dropin.PATCHED and hasattr(nb, name)
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)      # also where a GPU is present
    with pytest.raises(RuntimeError):
        dropin.patch(types.ModuleType("run_nerf"))        # no CUDA -> refuses


def test_bench_reference_arm_runs_on_cpu():
    import json, subprocess, sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600)
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["value"] > 0 and line["cpu_baseline"]["kind"] in ("reference", "port")
    assert line["steps"] >= 1 and abs(line["ms_per_step"] * 1e-3 * line["value"] - 4096) < 1.0     # measured, not extrapolated
    tr = line["cpu_baseline"].get("train")
    if line["cpu_baseline"]["kind"] == "reference":                                                 # SURVEY 8d: forward AND train beside the GPU numbers
        assert tr is not None and tr["value"] > 0 and abs(tr["ms_per_step"] * 1e-3 * tr["value"] - 4096) < 1.0


def _cuobjdump(*args):
    import shutil, subprocess
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe):
        pytest.skip("cuobjdump not available")
    from nerf_pytorch_b200 import _lib
    return subprocess.run([exe, *args, _lib.LIB_PATH], capture_output=True, text=True, timeout=600).stdout


def test_built_kernels_use_blackwell_tensor_and_tma_instructions(nb):
    """Static evidence in the cross-compiled sm_100a SASS (no GPU needed): the fused forward (inference and training
    instantiations) and the dgrad chain issue cta_group::2 tcgen05.mma, load weights with tensor-map TMA, read
    accumulators with tcgen05.ld and commit through multicast mbarrier arrives; the training-mode forward and the dgrad
    chain copy their tiles out with bulk stores (the inference instantiation has none); the weight-gradient kernel issues
    tcgen05.mma on bulk-loaded tiles.
    Guards against a silent regression to mma.sync / plain loads."""
    sass = _cuobjdump("-sass")
    funcs = {}
    cur = None
    for ln in sass.splitlines():
        m = re.search(r"Function : (\S+)", ln)
        if m:
            cur = m.group(1); funcs[cur] = []
        elif cur is not None:
            funcs[cur].append(ln)
    def body(sub):
        names = [k for k in funcs if sub in k]
        assert len(names) == 1, (sub, names)
        return "\n".join(funcs[names[0]])
    infer, train, dgrad, wgrad = body("march_tc2_kernelILb0"), body("march_tc2_kernelILb1"), body("dgrad_tc2_kernel"), body("wgrad_tc_kernel")
    for mnem in ("UTCHMMA.2CTA", "UTMALDG.2D.2CTA", "LDTM.x32", "UTCBAR.2CTA.MULTICAST", "SYNCS.PHASECHK.TRANS64.TRYWAIT", "ELECT", "F2FP.RELU"):
        assert mnem in infer and mnem in train, mnem
    for mnem in ("UTCHMMA.2CTA", "UTMALDG.2D.2CTA", "LDTM.x32", "UTCBAR.2CTA.MULTICAST", "ELECT", "F2FP.SATFINITE", "UBLKCP.G.S"):
        assert mnem in dgrad, mnem
    assert "UBLKCP.G.S" in train and "UBLKCP.G.S" not in infer          # shared -> global bulk stores: training mode only
    for mnem in ("UTCHMMA", "UBLKCP", "LDTM.x32", "UTCBAR"):
        assert mnem in wgrad, mnem
    for b in (infer, train, dgrad, wgrad):
        assert "HMMA.16816" not in b                                    # no mma.sync path


def test_fused_kernels_fit_their_resource_budget(nb):
    """640 threads x 96 registers is the whole register file; the fused kernels must not exceed it, and their spill
    stack stays small (sincosf slow path + the deferred raw values)."""
    usage = _cuobjdump("-res-usage")
    found = {}
    lines = usage.splitlines()
    for i, ln in enumerate(lines):
        m = re.search(r"Function (\S*(?:march_tc2|dgrad_tc2)_kernel\S*):", ln)
        if m and i + 1 < len(lines):
            r = re.search(r"REG:(\d+) STACK:(\d+)", lines[i + 1])
            found[m.group(1)] = (int(r.group(1)), int(r.group(2)))
    assert len(found) == 3, found
    for name, (reg, stack) in found.items():
        assert reg <= 96, (name, reg)
        assert stack <= 160, (name, stack)
