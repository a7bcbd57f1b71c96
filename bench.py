#!/usr/bin/env python
"""bench.py -- rays/sec of the NeRF ray-marching hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--mode forward|train] [--impl b200|reference|torch_gpu] [--dump-outputs DIR]

One "step" = one pass of the hot path over one 4096-ray batch of synthetic lego-shaped rays (BASELINE configs[1]:
64 coarse + 128 fine samples, 8x256 MLP + 128-wide view head).
  * headline (`value`, `e2e`, `roofline`): the FORWARD render_rays (render() under no_grad, test-time kwargs).  With N GPUs
    every rank renders its own 4096-ray batch ("scaling": "weak", no data-path collective).
  * `train`: the TRAIN step of run_nerf.py:760-784 (render with retraw, two MSE terms, backward, Adam, rate decay) through
    nerf_pytorch_b200.trainer.FusedTrainStep, device-resident and end to end (host rays + targets in, loss out), with the
    893 190 144 FLOP/ray roofline of SURVEY 8d; with N GPUs also `train_dp`: data parallel on a FIXED global 4096-ray batch
    (strong scaling, one all-reduce of the flat 4.77 MB gradient per step) and `frame`: an 800x800 frame ray-sharded over the
    ranks with the [rays,5] all-gather (BASELINE configs[3], [4]).
  * `torch_gpu` (N = 1): the UNMODIFIED reference (baseline/_ref/run_nerf.py: its own render(), autograd and Adam) on the
    same GPU, fp32 and TF32 matmuls, forward and train -- what the north star's ">= 10x" is relative to.
  * `cpu_baseline` / `--impl reference`: the reference on the host cores (the unmodified script when baseline/_ref is
    present -- kind "reference" --, else the op-chain port oracle/torch_ref.py -- kind "port").
JSON keys: see the build spec (value, e2e, roofline, cpu_baseline, clocks, gpu_launches ...).
--dump-outputs DIR writes what the last timed step of the headline path computed on rank 0 as DIR/<name>.npy (float32), so
that two builds can be compared output for output (the inputs are seeded: the same arguments give the same inputs).  Forward:
render()'s rgb_map, disp_map, acc_map and extras (rgb0, disp0, acc0, z_std), deterministic.  --mode train: the step's loss
(train_loss), the parameters after it (train_params) and its gradient (train_grads), flat in the networks' parameter order;
the backward accumulates with atomics, so these differ from run to run by rounding that the optimizer steps amplify.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time
import types

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
REF = os.path.join(ROOT, "baseline", "_ref")

N_RAYS, N_SAMPLES, N_IMPORTANCE = 4096, 64, 128
FLOP_PER_RAY_FWD = 303_824_896          # SURVEY 8d / Appendix B: 593 408 MAC x 2 x 256 evaluations
TRAIN_BYTES_PER_TILE = 1230848 + 1411072          # record bytes written + read per 128-row tile of a train step (DESIGN.md 9)
FLOP_PER_RAY_TRAIN = 893_190_144        # SURVEY 8d: forward + wgrad + dgrad (no recompute counted)
WORKLOAD = "lego 400x400 synthetic rays, N_rand=4096, N_samples=64 + N_importance=128, D=8 W=256 use_viewdirs, forward render_rays"
WORKLOAD_TRAIN = "lego 400x400 synthetic rays, N_rand=4096, 64+128 samples, D=8 W=256 use_viewdirs: render(retraw) + 2 x img2mse + backward + Adam + lr decay (run_nerf.py:760-784), perturb=1"


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        with open(path) as f:
            pk = json.load(f)
        return float(pk["bf16_tflops"]), "measured (MEASURED_PEAKS.json bf16_tflops, burst; fp16 == bf16 rate)", pk.get("bf16_tflops_sustained"), pk.get("hbm_gbs")
    return 1590.0, "fallback (B200_PROFILING.md 1.59 PFLOP/s)", None, 6650.0


# --------------------------------------------------------------------------------------------
# the unmodified reference (baseline/_ref), importable on CPU or GPU
# --------------------------------------------------------------------------------------------

def import_reference():
    """run_nerf from baseline/_ref with stand-ins for the two packages this image lacks (neither is on the path)."""
    if not os.path.isfile(os.path.join(REF, "run_nerf.py")):
        return None
    for name in ("imageio", "matplotlib", "matplotlib.pyplot", "configargparse"):
        sys.modules.setdefault(name, types.ModuleType(name))
    if REF not in sys.path:
        sys.path.insert(0, REF)
    import importlib
    return importlib.import_module("run_nerf")


def reference_setup(mod, device, tmpdir):
    """create_nerf() of the reference with the synthetic weights loaded -> (render_kwargs_train, render_kwargs_test, grad_vars, optimizer)"""
    import torch
    from oracle import synth
    os.makedirs(os.path.join(tmpdir, "bench"), exist_ok=True)
    args = argparse.Namespace(multires=10, multires_views=4, i_embed=0, use_viewdirs=True, N_importance=N_IMPORTANCE, N_samples=N_SAMPLES,
                              netdepth=8, netwidth=256, netdepth_fine=8, netwidth_fine=256, netchunk=65536, lrate=5e-4, basedir=tmpdir,
                              expname="bench", ft_path=None, no_reload=True, perturb=1.0, white_bkgd=True, raw_noise_std=0.0,
                              dataset_type="blender", no_ndc=False, lindisp=False)
    tr, te, start, grad_vars, opt = mod.create_nerf(args)
    for key, seed in (("network_fn", 0), ("network_fine", 1)):
        tr[key].load_state_dict({k: torch.from_numpy(v).to(device) for k, v in synth.nerf_state(seed).items()})
    for kw in (tr, te):
        kw.update(near=2., far=6.)
    return tr, te, grad_vars, opt


# --------------------------------------------------------------------------------------------
# CPU arm
# --------------------------------------------------------------------------------------------

def _cpu_limit():
    """Host threads this process may use: scheduler affinity capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            q, per = f.read().split()[:2]
        if q != "max":
            n = max(1, min(n, int(float(q) / float(per) + 0.5)))
    except (OSError, ValueError):
        pass
    return n


def cpu_rays_per_s(n_rays, reps, warmup, budget_s=45.0, train_step=False):
    """The reference's forward render of `n_rays` rays on the host cores: the unmodified script when baseline/_ref exists
    (kind "reference"), else the restated op chain (kind "port").  The thread count is calibrated ON THE REAL SAMPLE SIZE
    (more threads than the container owns slows torch's CPU ops down badly); time-bounded; returns the MEDIAN."""
    import tempfile
    import torch
    from oracle import synth
    sb = synth.ray_batch("lego", n_rays, seed=0)
    rays = torch.from_numpy(sb["rays"])
    mod = import_reference()
    train_fn = None
    if mod is not None and not torch.cuda.is_available():
        kind = "reference"
        tr, te, _, opt = reference_setup(mod, torch.device("cpu"), tempfile.mkdtemp())
        target = torch.rand(n_rays, 3, generator=torch.Generator().manual_seed(1))

        def train_fn():                                          # the body of train()'s step, run_nerf.py:760-776
            t0 = time.perf_counter()
            rgb, disp, acc, extras = mod.render(sb["H"], sb["W"], sb["K"], chunk=32768, rays=rays, verbose=False, retraw=True, **tr)
            opt.zero_grad()
            loss = mod.img2mse(rgb, target) + mod.img2mse(extras["rgb0"], target)
            loss.backward()
            opt.step()
            return time.perf_counter() - t0

        def run():
            t0 = time.perf_counter()
            with torch.no_grad():
                mod.render(sb["H"], sb["W"], sb["K"], chunk=32768, rays=rays, **te)
            return time.perf_counter() - t0
    else:
        kind = "port"
        from oracle import torch_ref as T
        sd = [{k: torch.from_numpy(v) for k, v in synth.nerf_state(s).items()} for s in (0, 1)]

        def run():
            t0 = time.perf_counter()
            with torch.no_grad():
                T.render(rays[0], rays[1], sd[0], sd[1], 2.0, 6.0, S=N_SAMPLES, n_imp=N_IMPORTANCE, white_bkgd=True)
            return time.perf_counter() - t0
    limit = _cpu_limit()
    best_t, best = None, None
    t_cal = time.perf_counter()
    for th in sorted({c for c in (8, 16, 32, 64, limit) if c <= limit}):
        torch.set_num_threads(th)
        dt = run()
        if best is None or dt < best:
            best_t, best = th, dt
        if time.perf_counter() - t_cal > budget_s / 2:
            break
    torch.set_num_threads(best_t)
    ts, t_start = [], time.perf_counter()
    for i in range(warmup + reps):
        dt = run()
        if i >= warmup:
            ts.append(dt)
        if ts and time.perf_counter() - t_start > budget_s:
            break
    sec = float(np.median(ts))
    train_sec = train_fn() if (train_step and train_fn is not None) else None      # ONE training step (SURVEY 8d: forward and train)
    return n_rays / sec, sec, best_t, kind, len(ts), train_sec


def reference_arm(args, rank):
    """`--impl reference`: the reference's own CPU implementation of the path on the host cores, all the threads it can use,
    each step the FULL 4096-ray batch when baseline/_ref is present (bounded by time: fewer steps, never a smaller batch)."""
    if rank != 0:
        return
    os.environ["CUDA_VISIBLE_DEVICES"] = ""                      # the reference picks cuda when it sees one (run_nerf.py:21)
    steps, warmup = max(1, args.steps), max(0, min(args.warmup, 1))
    import contextlib
    with contextlib.redirect_stdout(sys.stderr):                # the reference prints ('Found ckpts', 'Not ndc!'): stdout carries ONE JSON line
        rps, sec, threads, kind, done, train_sec = cpu_rays_per_s(N_RAYS, steps, warmup, budget_s=150.0, train_step=True)
    line = {"impl": "reference", "metric": "rays/sec", "value": rps, "unit": "rays/s", "n_gpus": args.gpus,
            "steps": done, "warmup": warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "steps_requested": steps, "note": "time-bounded: runs fewer steps than requested rather than a smaller batch"},
            "cpu_baseline": {"value": rps, "unit": "rays/s", "cores": threads, "kind": kind,
                             "sample": f"{N_RAYS} rays x (64+128) samples per step (the full batch), median of {done} step(s), "
                                       f"{'the unmodified run_nerf.render from baseline/_ref' if kind == 'reference' else 'torch fp32 CPU ops, the op chain of the reference (oracle/torch_ref.py)'}, "
                                       f"{threads} torch threads (calibrated on this batch; {os.cpu_count()} logical CPUs visible)",
                             "train": None if train_sec is None else {"value": N_RAYS / train_sec, "unit": "rays/s", "ms_per_step": train_sec * 1e3, "steps": 1,
                                                                       "what": "one step of the reference's loop body on the same threads: render(retraw=True), two img2mse, backward, Adam"}},
            "e2e": {"value": rps, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------
# the reference on the GPU (its own process: it relies on a CUDA default tensor type, run_nerf.py:876)
# --------------------------------------------------------------------------------------------

def torch_gpu_arm(args):
    import tempfile
    import torch
    from oracle import synth
    mod = import_reference()
    res = {"impl": "torch_gpu", "what": "the unmodified reference (baseline/_ref/run_nerf.py: render(), autograd, torch.optim.Adam) on cuda:0"}
    if mod is None or not torch.cuda.is_available():
        res["unavailable"] = "baseline/_ref or CUDA missing"
        print(json.dumps(res), flush=True)
        return
    torch.set_default_tensor_type("torch.cuda.FloatTensor")
    dev = torch.device("cuda:0")
    sb = synth.ray_batch("lego", N_RAYS, seed=0)
    rays = torch.from_numpy(sb["rays"]).to(dev)
    target = torch.rand(N_RAYS, 3)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    tmp = tempfile.mkdtemp()
    for tf32 in (False, True):
        torch.backends.cuda.matmul.allow_tf32 = tf32
        torch.backends.cudnn.allow_tf32 = tf32
        tr, te, grad_vars, opt = reference_setup(mod, dev, tmp)
        ms = []
        with torch.no_grad():
            for i in range(3 + 10):
                flush.zero_()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(); mod.render(sb["H"], sb["W"], sb["K"], chunk=32768, rays=rays, **te); b.record(); torch.cuda.synchronize()
                if i >= 3:
                    ms.append(a.elapsed_time(b))
        fwd = float(np.median(ms))
        ms = []
        for i in range(2 + 6):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            rgb, disp, acc, extras = mod.render(sb["H"], sb["W"], sb["K"], chunk=32768, rays=rays, verbose=False, retraw=True, **tr)
            opt.zero_grad()
            loss = mod.img2mse(rgb, target) + mod.img2mse(extras["rgb0"], target)
            loss.backward()
            opt.step()
            b.record(); torch.cuda.synchronize()
            if i >= 2:
                ms.append(a.elapsed_time(b))
        trn = float(np.median(ms))
        res["tf32" if tf32 else "fp32"] = {"forward_ms": fwd, "forward_rays_per_s": N_RAYS / (fwd * 1e-3), "train_ms": trn, "train_rays_per_s": N_RAYS / (trn * 1e-3)}
        del tr, te, grad_vars, opt
        torch.cuda.empty_cache()
    print(json.dumps(res), flush=True)


def _sub_json(argv, env=None, timeout=400):
    """run this script again with `argv`, return the last JSON line it prints (or an 'unavailable' record)"""
    try:
        e = dict(os.environ)
        for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT"):
            e.pop(k, None)
        if env:
            e.update(env)
        out = subprocess.run([sys.executable, os.path.abspath(__file__)] + argv, capture_output=True, text=True, timeout=timeout, env=e)
        for ln in reversed(out.stdout.strip().splitlines()):
            if ln.startswith("{"):
                return json.loads(ln)
        return {"unavailable": (out.stderr.strip().splitlines() or ["no output"])[-1][:300]}
    except Exception as ex:                                      # noqa: BLE001
        return {"unavailable": repr(ex)[:300]}


# --------------------------------------------------------------------------------------------
# clocks sampling
# --------------------------------------------------------------------------------------------

class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------

def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30, help="timed steps of each headline measurement")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "torch_gpu"])
    ap.add_argument("--mode", default="forward", choices=["forward", "train"], help="which measurement is the headline `value`")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-torch-gpu", action="store_true")
    ap.add_argument("--no-train", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        reference_arm(args, rank)
        return
    if args.impl == "torch_gpu":
        torch_gpu_arm(args)
        return
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    import __graft_entry__ as ge
    assert torch.cuda.is_available(), "bench.py needs a GPU (use --impl reference for the CPU arm)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    if rank == 0:
        ge.build()
    if world > 1:
        dist.barrier()
    import nerf_pytorch_b200 as nb
    from nerf_pytorch_b200 import _lib
    from nerf_pytorch_b200 import dist as nbdist
    from nerf_pytorch_b200.api import _QueryFn
    from nerf_pytorch_b200.trainer import FusedTrainStep
    from oracle import synth
    lib = _lib.load()
    peak, peak_src, peak_sus, hbm_gbs = load_peaks()

    def make_nets():
        nets = []
        for seed in (0, 1):
            m = nb.NeRF(D=8, W=256, input_ch=63, input_ch_views=27, output_ch=5, skips=[4], use_viewdirs=True)
            m.load_state_dict({k: torch.from_numpy(v) for k, v in synth.nerf_state(seed).items()})
            nets.append(m.to(dev))
        return nets

    nets = make_nets()
    e, _ = nb.get_embedder(10, 0)
    ed, _ = nb.get_embedder(4, 0)
    q = _QueryFn(e, ed, 65536, 10, 4, 0)
    sb = synth.ray_batch("lego", N_RAYS, seed=rank)
    kw = dict(ndc=False, near=2., far=6., use_viewdirs=True, network_fn=nets[0], network_fine=nets[1], network_query_fn=q,
              N_samples=N_SAMPLES, N_importance=N_IMPORTANCE, perturb=0., white_bkgd=True, raw_noise_std=0.)
    rays_host = torch.from_numpy(sb["rays"]).pin_memory()
    rays_dev = rays_host.to(dev)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)            # > 126 MB L2

    last = {}

    def timed(fn, steps, warmup, use_events=True):
        """-> (median ms per step, max over ranks); last["out"] is what the last timed call returned.  L2 flushed between
        timed iterations, outside the timed region."""
        for _ in range(warmup):
            flush.zero_(); fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        evs, walls = [], []
        for _ in range(steps):
            flush.zero_()
            if use_events:
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(); out = fn(); b.record()
                evs.append((a, b))
            else:
                torch.cuda.synchronize()
                t0 = time.perf_counter(); out = fn(); walls.append((time.perf_counter() - t0) * 1e3)
        last["out"] = out
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        per = [a.elapsed_time(b) for a, b in evs] if use_events else walls
        ms_med, ms_mean = float(np.median(per)), float(np.mean(per))
        if world > 1:
            t = torch.tensor([ms_med, ms_mean], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms_med, ms_mean = float(t[0].item()), float(t[1].item())
        return ms_med, ms_mean

    def read_timing():
        kms, kn, kfl = C.c_double(), C.c_int64(), C.c_double()
        kinds = (C.c_double * 3)()
        lib.nerf_b200_timing_read_kinds(C.byref(kms), C.byref(kn), C.byref(kfl), kinds)
        return kms.value, kn.value, kfl.value, [kinds[0], kinds[1], kinds[2]]

    sampler = ClockSampler(local_rank)
    sampler.start()

    # ---------------- forward ----------------
    def step_resident():
        with torch.no_grad():
            return nb.render(sb["H"], sb["W"], sb["K"], chunk=32768, rays=rays_dev, **kw)

    def step_eager_e2e():
        with torch.no_grad():
            rgb, disp, acc, _ = nb.render(sb["H"], sb["W"], sb["K"], chunk=32768, rays=rays_host.to(dev, non_blocking=True), **kw)
            out = torch.cat([rgb, disp[:, None], acc[:, None]], -1).to("cpu")
        return out

    graphed = nb.GraphedRender(sb["H"], sb["W"], sb["K"], N_RAYS, chunk=32768, **kw)
    step_resident(); torch.cuda.synchronize()
    l0 = nb.launch_count(); step_resident(); fwd_launches = nb.launch_count() - l0
    total_steps = args.warmup + args.steps
    lib.nerf_b200_timing_enable(1)
    ms_res, ms_res_mean = timed(step_resident, args.steps, args.warmup)
    dump_fwd, dump_train = {}, {}
    if args.dump_outputs:
        rgb, disp, acc, extras = last["out"]
        dump_fwd = {k: v.cpu().numpy() for k, v in dict(rgb_map=rgb, disp_map=disp, acc_map=acc, **extras).items()}
    kms, kn, kfl, _ = read_timing()                 # accumulators hold warm-up + timed launches: per-launch averages are reported
    lib.nerf_b200_timing_enable(0)
    ms_e2e, _ = timed(lambda: graphed(rays_host), args.steps, args.warmup, use_events=False)
    ms_e2e_eager, _ = timed(step_eager_e2e, max(5, args.steps // 3), 3, use_events=False)
    value = N_RAYS * world / (ms_res * 1e-3)
    achieved = (kfl / (kms * 1e-3)) / 1e12 if kms > 0 else 0.0
    traffic = None
    tfile = os.path.join(ROOT, "profiles", "march_tc_traffic.json")
    if os.path.isfile(tfile):
        with open(tfile) as f:
            traffic = json.load(f).get("dram_bytes_per_launch")
    fwd = {"value": value, "ms_per_step": ms_res, "ms_per_step_mean": ms_res_mean,
           "e2e": {"value": N_RAYS * world / (ms_e2e * 1e-3), "unit": "rays/s", "h2d_bytes_per_step": int(rays_host.numel() * 4),
                   "d2h_bytes_per_step": int(N_RAYS * 5 * 4), "ms_per_step": ms_e2e,
                   "api": "nerf_pytorch_b200.GraphedRender(...)(rays_host): H2D copy, CUDA-graph replay of render(), D2H copy of rgb/disp/acc, stream sync",
                   "eager_render": {"value": N_RAYS * world / (ms_e2e_eager * 1e-3), "ms_per_step": ms_e2e_eager,
                                    "api": "nerf_pytorch_b200.render(rays=host.to(device)) + .to('cpu'): the drop-in call itself"}},
           "roofline": {"bound": "tensor", "kernel": "march_tc2_kernel (cta_group::2 pair; coarse + fine launches)", "achieved": achieved, "peak": peak,
                        "unit": "TFLOP/s", "frac": achieved / peak if peak else None, "traffic": traffic, "peak_source": peak_src,
                        "peak_sustained": peak_sus, "frac_sustained": (achieved / peak_sus) if peak_sus else None,
                        "kernel_ms_per_step": kms / max(1, kn) * 2, "launches_timed": int(kn)},
           "gpu_launches": int(fwd_launches * args.steps)}

    # ---------------- train ----------------
    train = None
    extra = {}
    if not args.no_train:
        tkw = dict(kw)
        tkw.update(perturb=1.)
        tgt_host = torch.rand(N_RAYS, 3, generator=torch.Generator().manual_seed(1)).pin_memory()

        def run_train(n_local, group_world):
            tnets = make_nets()
            k2 = dict(tkw); k2.update(network_fn=tnets[0], network_fine=tnets[1])
            tr = FusedTrainStep(sb["H"], sb["W"], sb["K"], n_local, k2, lrate=5e-4, lrate_decay=250)
            lo = rank * n_local if group_world else 0
            r_h = rays_host[:, lo:lo + n_local].contiguous().pin_memory() if n_local != N_RAYS else rays_host
            t_h = tgt_host[lo:lo + n_local].contiguous().pin_memory() if n_local != N_RAYS else tgt_host
            tr.rays.copy_(r_h); tr.target.copy_(t_h)
            l0_ = nb.launch_count(); tr._pack_rays(); tr._fwd_bwd(); tr._adam(); launches = nb.launch_count() - l0_     # one eager step to count launches
            torch.cuda.synchronize()
            lib.nerf_b200_timing_enable(0)
            ms_dev, ms_dev_mean = timed(tr.step_device, args.steps, args.warmup)
            ms_host, _ = timed(lambda: tr(r_h, t_h), args.steps, args.warmup, use_events=False)
            if args.dump_outputs and not group_world:
                dump_train.update(train_loss=tr.state[0:1].cpu().numpy(), train_params=tr.flat_p.cpu().numpy(), train_grads=tr.flat_g.cpu().numpy())
            # kernel split of the step: an eager (un-graphed) pass with the library's event bracketing on
            lib.nerf_b200_timing_enable(1)
            for _ in range(3):
                tr._pack_rays(); tr._fwd_bwd(); tr._adam()
            torch.cuda.synchronize()
            kms_t, kn_t, kfl_t, kinds = read_timing()
            lib.nerf_b200_timing_enable(0)
            loss = float(tr.state[0].item())
            del tr
            torch.cuda.empty_cache()
            return ms_dev, ms_dev_mean, ms_host, launches, [k / 3 for k in kinds], loss

        ms_t, ms_t_mean, ms_t_host, t_launches, kinds, loss = run_train(N_RAYS, False)
        tval = N_RAYS * world / (ms_t * 1e-3)
        ach_t = N_RAYS * FLOP_PER_RAY_TRAIN / (ms_t * 1e-3) / 1e12
        train = {"metric": "rays/sec (train step)", "value": tval, "unit": "rays/s", "ms_per_step": ms_t, "ms_per_step_mean": ms_t_mean, "scaling": "weak",
                 "parallelism": "single GPU" if world == 1 else f"data parallel x{world}: 4096 rays per GPU (global batch {N_RAYS * world}), one all-reduce of the flat 4.77 MB gradient per step",
                 "workload": WORKLOAD_TRAIN, "loss": loss,
                 "e2e": {"value": N_RAYS * world / (ms_t_host * 1e-3), "unit": "rays/s", "ms_per_step": ms_t_host,
                         "h2d_bytes_per_step": int(rays_host.numel() * 4 + tgt_host.numel() * 4), "d2h_bytes_per_step": 16,
                         "api": "nerf_pytorch_b200.trainer.FusedTrainStep(...)(rays_host, target_host): H2D copies, ONE CUDA-graph replay (pack, forward in training mode, fused MSE seeds, tensor-core backward, flat Adam), D2H of the loss, stream sync"},
                 "gpu_launches_per_step": int(t_launches),
                 "roofline": {"bound": "tensor", "what": "whole train step: algorithmic 893 190 144 FLOP/ray (fwd + dgrad + wgrad, SURVEY 8d) over the step's device time",
                              "achieved": ach_t, "peak": peak, "unit": "TFLOP/s", "frac": ach_t / peak if peak else None, "peak_source": peak_src,
                              "kernel_ms_per_step": {"forward_passes_training_mode": kinds[0], "dgrad_chains": kinds[1], "wgrad": kinds[2]},
                              "kernel_ms_note": "split taken in a separate EAGER pass with CUDA events around each launch (3 steps, straight after the timed loops): "
                                                "the kernels run a few % slower there than inside the graph replay that `ms_per_step` times; use it for the shares",
                              "hbm": {"what": "bytes the step's design moves through HBM (DESIGN.md 9): per 128-row tile 1 230 848 B of records written (activations, "
                                              "masks, gradients) and 1 411 072 B read back (wgrad 1 310 720, dgrad 65 536, rgb head 34 816)",
                                      "bytes_per_step": TRAIN_BYTES_PER_TILE * N_RAYS * 256 // 128,
                                      "achieved_gbs": TRAIN_BYTES_PER_TILE * N_RAYS * 256 // 128 / (ms_t * 1e-3) / 1e9, "peak_gbs": hbm_gbs,
                                      "frac": (TRAIN_BYTES_PER_TILE * N_RAYS * 256 // 128 / (ms_t * 1e-3) / 1e9 / hbm_gbs) if hbm_gbs else None},
                              "note": "the step is bound by HBM (record traffic) and shared-memory bandwidth, not by the tensor pipe: wgrad streams 2 x 64 KB of "
                                      "fp16 tile images per tile-layer at 64 MAC/B (DESIGN.md 9)"}}
        if world > 1:
            # strong scaling: the SAME global 4096-ray batch split over the ranks, one flat all-reduce per step
            n_local = N_RAYS // world
            # correctness of the split, observed in this run: DP gradient (N/G rays per rank, loss scaled 1/G, all-reduce) vs the
            # full 4096-ray batch on one GPU, deterministic sampling
            ckw = dict(tkw); ckw.update(perturb=0.)
            cn1, cn2 = make_nets(), make_nets()
            k1 = dict(ckw); k1.update(network_fn=cn1[0], network_fine=cn1[1])
            k2 = dict(ckw); k2.update(network_fn=cn2[0], network_fine=cn2[1])
            t_full = FusedTrainStep(sb["H"], sb["W"], sb["K"], N_RAYS, k1, use_graph=False, data_parallel=False)
            t_dp = FusedTrainStep(sb["H"], sb["W"], sb["K"], n_local, k2, use_graph=False)
            rays0 = torch.from_numpy(synth.ray_batch("lego", N_RAYS, seed=0)["rays"]).to(dev)       # the same batch on every rank
            t_full.rays.copy_(rays0); t_full.target.copy_(tgt_host.to(dev))
            t_dp.rays.copy_(rays0[:, rank * n_local:(rank + 1) * n_local]); t_dp.target.copy_(tgt_host.to(dev)[rank * n_local:(rank + 1) * n_local])
            t_full._pack_rays(); t_dp._pack_rays(); t_full._fwd_bwd(); t_dp._fwd_bwd()
            dist.all_reduce(t_dp.flat_g, op=dist.ReduceOp.SUM)
            torch.cuda.synchronize()
            gd, gf = t_dp.flat_g.double(), t_full.flat_g.double()
            dp_check = {"grad_rel_l2_vs_single_gpu_full_batch": float((gd - gf).norm() / gf.norm()), "grad_cosine": float((gd @ gf) / (gd.norm() * gf.norm())),
                        "loss_dp_sum_over_ranks_vs_full": None}
            lsum = t_dp.state[0:1].clone() / world
            dist.all_reduce(lsum, op=dist.ReduceOp.SUM)
            dp_check["loss_dp_mean_over_ranks"] = float(lsum.item()); dp_check["loss_full_batch"] = float(t_full.state[0].item())
            del t_full, t_dp, cn1, cn2
            torch.cuda.empty_cache()
            ms_dp, ms_dp_mean, ms_dp_host, _, kinds_dp, _ = run_train(n_local, True)
            extra["train_dp"] = {"metric": "rays/sec (train step, data parallel, fixed global batch)", "value": N_RAYS / (ms_dp * 1e-3), "unit": "rays/s",
                                 "ms_per_step": ms_dp, "scaling": "strong", "global_batch": N_RAYS, "rays_per_gpu": n_local,
                                 "collective": "one ncclAllReduce(SUM) of the flat fp32 gradient buffer: 1 191 688 elements = 4.77 MB per step",
                                 "check": dp_check,
                                 "kernel_ms_per_step": {"forward_passes_training_mode": kinds_dp[0], "dgrad_chains": kinds_dp[1], "wgrad": kinds_dp[2]}}
            # full-frame render, ray-sharded, all-gather of [rays, 5]
            Hf = Wf = 800
            focal = 0.5 * Wf / np.tan(0.5 * 0.6911112070083618)
            Kf = np.array([[focal, 0, 0.5 * Wf], [0, focal, 0.5 * Hf], [0, 0, 1]])
            c2w = torch.from_numpy(np.asarray(sb["c2w"], np.float32))
            if True:
                from nerf_pytorch_b200 import api as nbapi
                n_pix = Hf * Wf
                lo, hi = nbdist.shard_bounds(n_pix, rank, world)

                def frame():
                    with torch.no_grad():
                        packed = torch.empty((hi - lo, 11), device=dev)
                        cam = nbapi._camera(Hf, Wf, Kf, c2w)
                        _lib.check(lib.nerf_b200_pack_rays(None, None, None, C.byref(cam), hi - lo, lo, 0, 2.0, 6.0, 1, nbapi._ptr(packed), nbapi._stream(packed)), "pack_rays")
                        ret = nb.batchify_rays(packed, 32768, **{k: v for k, v in kw.items() if k not in ("ndc", "near", "far", "use_viewdirs")})
                        loc = torch.cat([ret["rgb_map"], ret["disp_map"][:, None], ret["acc_map"][:, None]], -1)
                        return nbdist.gather_pixels(loc, n_pix)
                full = frame()
                fcheck = None
                if rank == 0:                                   # the gathered frame vs rank 0 rendering every ray itself
                    with torch.no_grad():
                        rgb1, disp1, acc1, _ = nb.render(Hf, Wf, Kf, chunk=32768, c2w=c2w, **kw)
                    one = torch.cat([rgb1.reshape(-1, 3), disp1.reshape(-1, 1), acc1.reshape(-1, 1)], -1)
                    fcheck = float((torch.nan_to_num(full) - torch.nan_to_num(one)).abs().max().item())
                ms_f, _ = timed(frame, max(3, args.steps // 5), 2)
                extra["frame"] = {"metric": "rays/sec (800x800 frame, ray-sharded render + all-gather)", "value": n_pix / (ms_f * 1e-3), "unit": "rays/s",
                                  "ms_per_frame": ms_f, "scaling": "strong", "rays_per_frame": n_pix, "max_abs_diff_vs_single_gpu_render": fcheck,
                                  "collective": "all_gather of [rays/G, 5] fp32 stripes = 12.8 MB per frame; rays generated per rank from the 72-byte camera (pixel0 offset), no scatter"}
    clocks = sampler.stop()

    headline = fwd if args.mode == "forward" or train is None else None
    line = {
        "metric": "rays/sec" if headline is not None else "rays/sec (train step)",
        "value": fwd["value"] if headline is not None else train["value"], "unit": "rays/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": fwd["ms_per_step"] if headline is not None else train["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f16", "data": "synthetic",
        "config": {"workload": WORKLOAD if headline is not None else WORKLOAD_TRAIN, "rays_per_gpu_per_step": N_RAYS,
                   "operands": "fp16 x fp16 -> fp32 accumulate (tcgen05 kind::f16); backward: loss-scaled fp16 activation gradients",
                   "l2": "flushed between timed iterations (512 MiB memset, outside the timed events)",
                   "statistic": "median over the timed steps (mean reported beside it)",
                   "parallelism": f"ray-parallel x{world}, no data-path collective"},
        "e2e": fwd["e2e"] if headline is not None else train["e2e"],
        "gpu_launches": fwd["gpu_launches"] if headline is not None else int(train["gpu_launches_per_step"] * args.steps),
        "roofline": fwd["roofline"] if headline is not None else train["roofline"],
        "clocks": clocks,
    }
    if headline is not None and train is not None:
        line["train"] = train
    if headline is None:
        line["forward"] = fwd
    line.update(extra)
    if rank == 0 and world == 1:
        if not args.no_torch_gpu:
            line["torch_gpu"] = _sub_json(["--impl", "torch_gpu"], timeout=300)
            tg = line["torch_gpu"]
            if "tf32" in tg:
                line["torch_gpu"]["speedup"] = {"forward_vs_tf32": fwd["value"] / tg["tf32"]["forward_rays_per_s"], "forward_vs_fp32": fwd["value"] / tg["fp32"]["forward_rays_per_s"]}
                if train is not None:
                    line["torch_gpu"]["speedup"].update(train_vs_tf32=train["value"] / tg["tf32"]["train_rays_per_s"], train_vs_fp32=train["value"] / tg["fp32"]["train_rays_per_s"])
        if not args.no_cpu:
            ref = _sub_json(["--impl", "reference", "--steps", "3", "--warmup", "1"], env={"CUDA_VISIBLE_DEVICES": ""}, timeout=400)
            line["cpu_baseline"] = ref.get("cpu_baseline", ref)
    if rank == 0:
        if args.dump_outputs:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for k, v in (dump_fwd if headline is not None else dump_train).items():
                np.save(os.path.join(args.dump_outputs, k + ".npy"), v.astype(np.float32))
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
