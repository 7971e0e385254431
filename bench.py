#!/usr/bin/env python
"""bench.py — headline measurement of the B200-native HyperNeRF per-ray hot path.

Workload (BASELINE.json configs[1]): HyperNeRF translation warp + bendy sheet (hyper_dim 2), 64 coarse + 64 fine
samples, ONE training step = forward + MSE loss + backward over a 65 536-ray batch of synthetic LLFF-shaped rays
(strong scaling: the global batch is fixed and sharded over N GPUs, one NCCL all-reduce of the flat 5.9 MB gradient
per step), plus the Adam update.  Metric: train rays/s.

    python bench.py --gpus 1 --steps 5 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...
    python bench.py --impl reference        # the reference's CPU path on the host cores (live reference if reachable, else the pinned port)

One JSON line on stdout (rank 0).  See DESIGN.md "Measurement" for every field.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GLOBAL_RAYS = 65536
N_COARSE, N_FINE = 64, 64
SE3_FLOP_PER_EVAL = 2 * 857728            # SURVEY.md §8(d) config 5: SE3Field 144 128 + template (167-wide input) 713 600 MAC
SE3_TRUNK_FLOP_PER_EVAL = 2 * 713600
EMB = {'warp': list(range(100)), 'camera': [0], 'appearance': list(range(100)), 'time': list(range(100))}
SE3_KW = dict(near=0., far=1., n_samples_coarse=128, n_samples_fine=128, noise_std=1.0, use_warp=True, use_nerf_embed=False,
              use_alpha_cond=False, use_rgb_cond=False, hyper_slice_method='axis_aligned_plane', hyper_slice_out_dim=8,
              GLO_dim=8, share_GLO=True, xyz_fourier_dim=10, hyper_fourier_dim=6, view_fourier_dim=6, warp_field_type='se3')
FWD_FLOP_PER_EVAL = 2 * 801536            # SURVEY.md §8(d): 801 536 MAC per sample evaluation (unpadded)
TRUNK_FLOP_PER_EVAL = 2 * 673664          # the same without TranslationField (100 480) and HyperSheetMLP (27 392)
EVALS_PER_RAY = N_COARSE + (N_COARSE + N_FINE)
METRIC = "train rays/s (fwd+bwd, 64+64 samples/ray, HyperNeRF warp+bendy-sheet)"
WORKLOAD = "cfg2: HyperNeRF translation warp + bendy_sheet (hyper_dim 2), 65536-ray train batch, 64 coarse + 64 fine"


# --------------------------------------------------------------------------------------------------------------
# CPU baseline: the reference's own per-ray path on the host cores, on a bounded sample of each workload.
# The live, unmodified reference is used when its tree is reachable (oracle/ref_loader.py: $HN_REFERENCE_DIR, /root/reference,
# baseline/_ref) -> kind "reference"; on the GPU box, where a Python reference cannot travel, the pinned restatement
# (oracle/, checked against the live reference and its goldens by tests/test_oracle.py) -> kind "port".
# --------------------------------------------------------------------------------------------------------------
def _cpu_setup():
    from oracle import ref_loader
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    return cores, ref_loader.reference_available()


def _draws(n_rays, n_fine, it, noise=True):
    g = torch.Generator().manual_seed(it)
    d = dict(u_coarse=torch.rand(n_rays, N_COARSE, generator=g),
             noise_coarse=torch.randn(n_rays, N_COARSE, 1, generator=g) if noise else None,
             u_fine=torch.rand(n_rays, n_fine, generator=g),
             noise_fine=torch.randn(n_rays, N_COARSE + n_fine, 1, generator=g) if noise else None)
    return d


def cpu_reference_rate(n_rays=1024, repeats=2, warmup=1, workload="train"):
    """rays/s of the reference path on the host CPU.  workload: 'train' (cfg2 shape: 64+64, fwd + loss + bwd), 'render'
    (cfg3: 64+128, no_grad forward), 'static' (cfg4: models/nerf.py x2 + render_rays, 128+128, fwd + bwd), 'se3' (cfg5:
    SE3Field + axis-aligned slicing, 128+128, fwd + loss + bwd — always the restatement: the reference cannot run it)."""
    from hypernerf_torch_b200 import synthetic
    from oracle import hypernerf_oracle as orc
    from oracle import ref_loader, static_oracle
    cores, live = _cpu_setup()
    kind = "reference" if live else "port"
    rays, rgbs = synthetic.train_rays(n_rays, seed=0)
    n_fine = {"train": N_FINE, "render": 128, "static": 128, "se3": 128}[workload]
    if workload == "se3":
        from hypernerf_torch_b200.models import NerfModel
        live, kind = False, "port"
        shapes = {k: tuple(v.shape) for k, v in NerfModel(EMB, **SE3_KW).state_dict().items()}   # parameter containers only
        sd = {k: v.clone().requires_grad_(True) for k, v in synthetic.make_state_dict(shapes, seed=0, boosted=False).items()}
        cfg = orc.cfg_from_kwargs(SE3_KW)

        def step(it):
            for v in sd.values():
                v.grad = None
            g = torch.Generator().manual_seed(it)
            draws = dict(u_coarse=torch.rand(n_rays, 128, generator=g), noise_coarse=torch.randn(n_rays, 128, 1, generator=g),
                         u_fine=torch.rand(n_rays, 128, generator=g), noise_fine=torch.randn(n_rays, 256, 1, generator=g))
            out = orc.forward(sd, rays[:, :3], rays[:, 3:6], rays[:, 8].long(), draws, cfg)
            orc.mse_loss(out, rgbs).backward()
        what = "cfg5 SE3 warp + axis-aligned slicing (128+128 samples, fwd+loss+bwd; batched restatement)"
    elif workload == "static":
        sds = [synthetic.make_state_dict(synthetic.static_state_dict_shapes(), seed=i) for i in range(2)]
        if live:
            ref_loader.load_reference()
            from models.nerf import Embedding, NeRF            # the reference's own modules (sys.path set by the loader)
            from models.rendering import render_rays as ref_render_rays
            models = [NeRF(), NeRF()]
            for m, sd in zip(models, sds):
                m.load_state_dict(sd)
            emb = [Embedding(3, 10), Embedding(3, 4)]

            def step(it):
                for m in models:
                    m.zero_grad(set_to_none=True)
                torch.manual_seed(it)
                out = ref_render_rays(models, emb, rays[:, :8].contiguous(), N_samples=128, perturb=1.0, noise_std=1.0,
                                      N_importance=128, chunk=1 << 15)
                (torch.nn.functional.mse_loss(out['rgb_coarse'], rgbs) + torch.nn.functional.mse_loss(out['rgb_fine'], rgbs)).backward()
        else:
            sds = [{k: v.clone().requires_grad_(True) for k, v in sd.items()} for sd in sds]

            def step(it):
                g = torch.Generator().manual_seed(it)
                draws = dict(u_perturb=torch.rand(n_rays, 128, generator=g), noise_coarse=torch.randn(n_rays, 128, generator=g),
                             u_pdf=torch.rand(n_rays, 128, generator=g), noise_fine=torch.randn(n_rays, 256, generator=g))
                for sd in sds:
                    for v in sd.values():
                        v.grad = None
                out = static_oracle.render_rays(sds, rays[:, :8], draws, n_samples=128, n_importance=128)
                (torch.nn.functional.mse_loss(out['rgb_coarse'], rgbs) + torch.nn.functional.mse_loss(out['rgb_fine'], rgbs)).backward()
        what = "cfg4 static NeRF (128+128 samples, fwd+bwd)"
    else:
        train = workload == "train"
        sd = synthetic.make_state_dict(synthetic.cfg1_state_dict_shapes(), seed=0, boosted=False)
        if live:
            model = ref_loader.build_reference_model(seed=0, n_samples_fine=n_fine, noise_std=1.0 if train else None)
            model.load_state_dict(sd)

            def step(it):
                model.zero_grad(set_to_none=True)
                torch.manual_seed(it)
                with torch.set_grad_enabled(train):
                    out, _ = ref_loader.run_reference(model, rays)
                    if train:
                        (torch.nn.functional.mse_loss(out['coarse']['rgb'], rgbs) +
                         torch.nn.functional.mse_loss(out['fine']['rgb'], rgbs)).backward()
        else:
            sd = {k: v.clone().requires_grad_(train) for k, v in sd.items()}
            cfg = orc.default_cfg(n_fine=n_fine, noise_std=1.0 if train else 0.0)

            def step(it):
                for v in sd.values():
                    v.grad = None
                with torch.set_grad_enabled(train):
                    out = orc.forward(sd, rays[:, :3], rays[:, 3:6], rays[:, 8].long(), _draws(n_rays, n_fine, it, noise=train), cfg)
                    if train:
                        orc.mse_loss(out, rgbs).backward()
        what = "cfg2 train step (64+64 samples, fwd+loss+bwd)" if train else "cfg3 render (64+128 samples, no_grad forward)"
    best = float("inf")
    for it in range(warmup + repeats):
        t0 = time.perf_counter()
        step(it)
        dt = time.perf_counter() - t0
        if it >= warmup:
            best = min(best, dt)
    impl = "the unmodified reference imported in place" if live else "oracle port of the reference (a Python reference cannot travel to the GPU box)"
    if workload == "se3":
        impl = "batched restatement under oracle/ (the reference defines SE3Field but cannot run it: SURVEY.md §8(c))"
    return {"value": n_rays / best, "unit": "rays/s", "cores": cores, "kind": kind,
            "sample": f"{n_rays} rays of {what}, fp32 torch on {cores} CPU threads, {impl}, best of {repeats}"}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = max(1, min(args.steps, 5))
    cpu = cpu_reference_rate(n_rays=1024, repeats=steps, warmup=min(args.warmup, 1), workload="train")
    rate = cpu["value"]
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": "rays/s", "n_gpus": args.gpus, "steps": steps,
        "warmup": min(args.warmup, 1), "ms_per_step": 1e3 * 1024 / rate, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "note": "CPU arm: each step is a 1024-ray sample of the workload"},
        "cpu_baseline": cpu,
        "e2e": {"value": rate, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# --------------------------------------------------------------------------------------------------------------
# clocks
# --------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons DURING the timed region: an NVML polling thread (first sample at once, then every
    20 ms, so even the 65 ms timed region of the 8-GPU run is covered); nvidia-smi -lms as the fallback."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    MASKS = (("sw_power_cap", 0x4), ("hw_slowdown", 0x8), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40))

    def __init__(self, gpu_index):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
        try:
            gpu_index = int(vis.split(",")[gpu_index]) if vis else gpu_index
        except (ValueError, IndexError):
            pass
        self.rows, self.proc, self.idx = [], None, gpu_index
        self.sm, self.mx, self.reasons = [], [], set()
        self.nvml, self.handle, self.stop_flag, self.thread = None, None, threading.Event(), None

    def _poll(self):
        n = self.nvml
        reasons_fn = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
            getattr(n, "nvmlDeviceGetCurrentClocksThrottleReasons", None)
        while True:
            try:
                self.sm.append(float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)))
                if reasons_fn is not None:
                    bits = int(reasons_fn(self.handle))
                    for name, mask in self.MASKS:
                        if bits & mask:
                            self.reasons.add(name)
            except Exception:
                pass
            if self.stop_flag.wait(0.02):
                return

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self.idx)
            self.mx.append(float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)))
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.nvml is not None:
            self.stop_flag.set()
            self.thread.join(timeout=1.0)
            sm = sorted(self.sm)
            return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(self.mx) if self.mx else None,
                    "reasons": sorted(self.reasons), "samples": len(sm), "source": "nvml"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi"}


# --------------------------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------------------------
# Algorithmic work per sample evaluation (SURVEY.md §8(d), unpadded MACs x 2): which figure a profiled kernel launch counts
STATIC_FLOP_PER_EVAL = 2 * 593408         # models/nerf.py NeRF(D=8, W=256): 593 408 MAC per sample
# stash bytes the weight-gradient kernel streams per sample (design traffic, DESIGN.md §3): X slabs + dY slabs, read once
WGRAD_STASH_BYTES = {"mlp_wgrad": 8640 + 8288, "mlp_wgrad_trunk": 6176 + 5952}


def kernel_table(prof, secs, flop_full, flop_trunk):
    """Per-kernel totals of the CUDA-event pairs recorded around every MLP launch of a timed region (_lib.timed)."""
    per = {}
    for name, n, a, b in prof or []:
        d = per.setdefault(name, [0.0, 0, 0])
        d[0] += a.elapsed_time(b) / 1e3; d[1] += 1; d[2] += n
    kernels, executed = {}, 0.0
    for name, (t, cnt, nsamp) in per.items():
        # fwd, dgrad and wgrad each count 1x the forward FLOPs of the samples they process (bwd = 2x fwd)
        flops = (flop_trunk if name.endswith("_trunk") else flop_full) * nsamp
        executed += flops
        kernels[name] = {"launches": cnt, "seconds": t, "samples": nsamp, "tflops": flops / t / 1e12 if t > 0 else None,
                         "share_of_region": t / (secs if secs > 0 else 1)}
        if name in WGRAD_STASH_BYTES and t > 0:
            kernels[name]["stash_gbs"] = WGRAD_STASH_BYTES[name] * nsamp / t / 1e9
    return kernels, executed


def roofline_of(kernels, executed, secs, peaks, traffic_json, ms_key="avg_launch_ms"):
    """`roofline` object of one leg: the dominant MLP kernel (by summed CUDA-event time inside the timed region) against
    the roofline SURVEY.md §8(d) names for the MLP stack — dense bf16 tensor throughput on UNPADDED algorithmic FLOPs.
    The HBM view of the weight-gradient kernel (which streams this design's activation stashes) is kept next to it as
    `hbm_view`, and the whole region's executed-FLOP rate as `step_tensor_frac` (the north-star utilisation figure)."""
    if not kernels:
        return None
    peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
    peak_hbm = peaks.get("hbm_gbs", 6650.0)
    src = ("MEASURED_PEAKS.json: bf16_tflops_sustained (kernels timed inside a long step), hbm_gbs" if peaks else
           "fallback 1.4 PFLOP/s sustained, 6.65 TB/s (B200_PROFILING.md)")
    dom = max(kernels, key=lambda k: kernels[k]["seconds"])
    k = kernels[dom]
    traffic = None
    tr = traffic_json.get(dom)
    if tr:
        traffic = tr["dram_bytes_per_sample"] * k["samples"] / k["launches"]     # ncu dram bytes per launch
    roof = {"kernel": dom, "bound": "tensor", "achieved": k["tflops"], "peak": peak_tf, "unit": "TFLOP/s",
            "frac": k["tflops"] / peak_tf, "traffic": traffic, "peak_source": src,
            ms_key: 1e3 * k["seconds"] / k["launches"],
            "algorithmic_flop_per_launch": k["tflops"] * 1e12 * k["seconds"] / k["launches"],
            "step_tensor_frac": (executed / secs / 1e12) / peak_tf, "executed_tflops_per_gpu": executed / secs / 1e12,
            "kernels": kernels}
    wg = [n for n in kernels if n in WGRAD_STASH_BYTES]
    if wg:
        n = max(wg, key=lambda x: kernels[x]["seconds"])
        roof["hbm_view"] = {"kernel": n, "bound": "hbm", "achieved": kernels[n]["stash_gbs"], "peak": peak_hbm, "unit": "GB/s",
                            "frac": kernels[n]["stash_gbs"] / peak_hbm,
                            "note": "bytes are this design's stash traffic (X + dY slabs read once), not algorithmic bytes of "
                                    "the reference path: explains the tensor fraction, does not replace it"}
    return roof


def run_gpu_arm(args):
    import torch.distributed as dist
    from hypernerf_torch_b200 import _lib, ray_utils, synthetic
    from hypernerf_torch_b200 import train as hn_train
    from hypernerf_torch_b200.models import NerfModel

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback (use --impl reference)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _lib.lib()  # fail loudly if the native library is missing

    peaks, traffic_json = {}, {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    try:
        traffic_json = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json")))
    except Exception:
        pass

    emb = EMB
    model = NerfModel(emb, near=0., far=1., n_samples_coarse=N_COARSE, n_samples_fine=N_FINE, noise_std=1.0,
                      hyper_slice_method='bendy_sheet', hyper_slice_out_dim=2, use_warp=True, use_nerf_embed=False,
                      use_alpha_cond=False, use_rgb_cond=False, GLO_dim=8, share_GLO=True, xyz_fourier_dim=10,
                      hyper_fourier_dim=6, view_fourier_dim=6)
    model.load_state_dict(synthetic.make_state_dict(model, seed=0, boosted=False))
    model = model.to(dev)
    fg = hn_train.FlatGrads(model.parameters())
    model.attach_flat_grads(fg)

    rays_all, rgbs_all = synthetic.train_rays(GLOBAL_RAYS, seed=0)
    # one-shot check before anything is timed: the N-GPU step (ray shards, rank-sliced global draws, one flat all-reduce)
    # reproduces the 1-GPU step on the same 4 096 rays (SURVEY.md §8(e)); raises if it does not
    dp_parity = None
    if world > 1:
        dp_parity = {"rays": 4096, "tol": 1e-4,
                     "rel_l2": hn_train.dp_parity_check(model, fg, rays_all[:4096].to(dev), rgbs_all[:4096].to(dev), tol=1e-4)}
    opt = hn_train.FusedAdam(fg, lr=5e-4, eps=1e-8)   # Adam of utils/__init__.py:29-31 / opt.py:53-56, one launch
    # Every timed step trains from this initial state (weights, Adam moments and step count, restored outside the events).
    # The backward kernels reduce with float atomics, so a step is reproducible only up to rounding, and a chain of Adam
    # steps amplifies that rounding until two runs train different models; from one fixed state, the same arguments give
    # the same outputs from run to run.
    params0 = opt.flat.clone()
    opt_state0 = {k: v.clone() if torch.is_tensor(v) else v for k, v in opt.state_dict().items()}

    @torch.no_grad()
    def restore_train_state():
        opt.flat.copy_(params0)
        torch.autograd.graph.increment_version(fg.params)   # the models' packed-weight caches key on the version counters
        opt.load_state_dict(opt_state0)

    # inputs: this rank's contiguous shard of the global batch, resident in HBM (value) and in pinned host memory (e2e)
    lo, hi = hn_train.shard_bounds(GLOBAL_RAYS, rank, world)
    rays_h = rays_all[lo:hi].contiguous().pin_memory()
    rgbs_h = rgbs_all[lo:hi].contiguous().pin_memory()
    rays_d, rgbs_d = rays_h.to(dev), rgbs_h.to(dev)
    chunk = args.chunk
    l2_flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2

    def step(rays, rgbs):
        return hn_train.train_step(model, rays, rgbs, fg, global_rays=GLOBAL_RAYS, chunk=chunk, optimizer=opt)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    torch.manual_seed(1234 + rank)
    for _ in range(max(args.warmup, 3)):
        step(rays_d, rgbs_d)
    sync_all()

    def timed_loop(fn, steps, profile=False, before=None):
        """EXACTLY `steps` steps; device time by CUDA events on the launching stream, `before` and an L2 flush between
        steps (outside the events); returns (seconds summed over steps, max over ranks; launches; per-kernel events)."""
        evs = []
        launches0 = _lib.launches
        if profile:
            _lib.profile = []
        sync_all()
        for _ in range(steps):
            if before is not None:
                before()
            l2_flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            evs.append((e0, e1))
        sync_all()
        secs = sum(a.elapsed_time(b) for a, b in evs) / 1e3
        prof, _lib.profile = _lib.profile, None
        t = torch.tensor([secs], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), _lib.launches - launches0, prof

    last = {}

    def timed_step():
        last["loss"] = step(rays_d, rgbs_d)

    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    secs, launches, prof = timed_loop(timed_step, args.steps, profile=True, before=restore_train_state)
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        # what a caller of the train step holds after the last timed step, before the other legs train further: the loss,
        # the all-reduced gradient and the Adam-updated parameters (flat buffers, FlatGrads order incl. padding; 5.9 MB each)
        dump_outputs(args.dump_outputs, {"loss": last["loss"], "grads": fg.flat, "params": opt.flat})

    # end to end: host rows in, loss out, every step
    loss_h = torch.empty((), dtype=torch.float32).pin_memory()

    # The end-to-end caller synchronises every step (it reads the loss), so the host's ~45 launches per chunk are exposed
    # once a step is short (N = 8: 11 ms): the chunk loop is captured in a CUDA graph (train.GraphedTrainStep); the exchange
    # and the optimizer launch stay eager.  Falls back to the eager step if the capture is refused.
    gstep, graph_note = None, "eager"
    if not args.no_graph:
        try:
            # (the graph's private memory pool keeps every stash of a chunk allocated for the graph's lifetime: the eager
            # leg's pool is released first; 16 384-ray chunks: 0.3 % behind the eager `value` on one box, 8 192: 0.7 %)
            gchunk = min(chunk, args.graph_chunk)
            torch.cuda.empty_cache()          # the eager leg's pool goes back before the graph builds its own
            gstep = hn_train.GraphedTrainStep(model, fg, hi - lo, GLOBAL_RAYS, gchunk)
            gstep(rays_d, rgbs_d, opt)
            torch.cuda.synchronize()
            graph_note = f"chunk loop replayed from a CUDA graph ({gstep.launches} captured launches, {gchunk}-ray chunks)"
        except Exception as e:   # noqa: BLE001 - any capture failure: measure eagerly and say so
            gstep, graph_note = None, f"eager (graph capture failed: {type(e).__name__})"
            torch.cuda.synchronize()

    def e2e_step():
        r = rays_h.to(dev, non_blocking=True)
        c = rgbs_h.to(dev, non_blocking=True)
        loss = gstep(r, c, opt) if gstep is not None else step(r, c)
        loss_h.copy_(loss, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    e2e_step()
    secs_e2e, _, _ = timed_loop(e2e_step, args.steps)
    use_graph = gstep is not None
    gstep = None                      # the graph's private pool goes back before the other legs allocate
    torch.cuda.empty_cache()
    kernels, executed = kernel_table(prof, secs, FWD_FLOP_PER_EVAL, TRUNK_FLOP_PER_EVAL)
    roof = roofline_of(kernels, executed, secs, peaks, traffic_json)
    if roof:
        roof["executed_mflop_per_ray"] = executed / (args.steps * GLOBAL_RAYS / world) / 1e6

    # ---------------------------------------------------------------------------------------------------------------
    # secondary metric of BASELINE.json ("render Mrays/s", configs[2]): 1008x756 frames, 64+128 samples, no_grad,
    # random-init weights, rows of the frame sharded over the ranks (no collective); device time, max over ranks.
    #   value: the frame's ray rows resident in HBM;
    #   e2e:   per frame a camera pose comes from the host (48 bytes), the rays are generated on the device
    #          (hn_make_ndc_rays), rendered, and the rgb image goes back to pinned host memory.
    # ---------------------------------------------------------------------------------------------------------------
    render = None
    if not args.no_render:
        rmodel = NerfModel(emb, near=0., far=1., n_samples_coarse=64, n_samples_fine=128, noise_std=None,
                           hyper_slice_method='bendy_sheet', hyper_slice_out_dim=2, use_warp=True, use_nerf_embed=False,
                           use_alpha_cond=False, use_rgb_cond=False, GLO_dim=8, share_GLO=True, xyz_fourier_dim=10,
                           hyper_fourier_dim=6, view_fourier_dim=6)
        rmodel.load_state_dict(model.state_dict())
        rmodel = rmodel.to(dev).eval()
        Hh, Ww = synthetic.H, synthetic.W
        n_frame = Hh * Ww
        flo, fhi = hn_train.shard_bounds(n_frame, rank, world)
        frame_d = synthetic.frame_rays(image_id=3, seed=0)[flo:fhi].contiguous().to(dev)
        frames = max(5, args.render_frames)
        hn_train.render_rays(rmodel, frame_d, chunk=args.render_chunk)       # warm-up: one whole frame (allocator, clocks)
        secs_r, launches_r, prof_r = timed_loop(lambda: hn_train.render_rays(rmodel, frame_d, chunk=args.render_chunk), frames, profile=True)
        img_h = torch.empty(fhi - flo, 3, dtype=torch.float32).pin_memory()
        poses = [torch.tensor([[1., 0., 0., 0.02 * i], [0., 1., 0., -0.01 * i], [0., 0., 1., 0.0]]) for i in range(frames)]
        it = iter(range(10 ** 9))

        def render_e2e():
            c2w = poses[next(it) % frames]
            rows = ray_utils.frame_rays_ndc(Hh, Ww, synthetic.FOCAL, c2w, image_id=3, device=dev)[flo:fhi]
            out = hn_train.render_rays(rmodel, rows, chunk=args.render_chunk, keys=('rgb',))
            img_h.copy_(out['rgb'], non_blocking=True)
            torch.cuda.current_stream().synchronize()

        render_e2e()
        secs_re, _, _ = timed_loop(render_e2e, frames)
        rk, rexec = kernel_table(prof_r, secs_r, FWD_FLOP_PER_EVAL, TRUNK_FLOP_PER_EVAL)
        render = {"value": n_frame * frames / secs_r / 1e6, "unit": "Mrays/s", "rays_per_frame": int(n_frame),
                  "samples": "64+128", "ms_per_frame": 1e3 * secs_r / frames, "frames_timed": frames,
                  "e2e": {"value": n_frame * frames / secs_re / 1e6, "unit": "Mrays/s", "h2d_bytes_per_step": 48,
                          "d2h_bytes_per_step": int(img_h.numel() * 4), "ms_per_frame": 1e3 * secs_re / frames,
                          "note": "pose in (host), rays generated on the device, rgb image out (pinned host)"},
                  "gpu_launches": launches_r, "roofline": roofline_of(rk, rexec, secs_r, peaks, traffic_json),
                  "workload": "cfg3: full-frame eval render 1008x756, random-init weights, no_grad"}
        del rmodel, frame_d
        torch.cuda.empty_cache()

    # ---------------------------------------------------------------------------------------------------------------
    # secondary workload (BASELINE.json configs[3]): static NeRF baseline (models/nerf.py x2 + render_rays), 262 144-ray
    # batch sharded over the ranks, 128+128 samples, perturb=1, noise_std=1, forward + backward (no optimizer)
    # ---------------------------------------------------------------------------------------------------------------
    static = None
    if not args.no_static:
        from hypernerf_torch_b200.nerf import Embedding, NeRF
        from hypernerf_torch_b200.rendering import render_rays as static_render_rays
        smodels = [NeRF().to(dev), NeRF().to(dev)]
        semb = [Embedding(3, 10), Embedding(3, 4)]
        n_static = 262144
        slo, shi = hn_train.shard_bounds(n_static, rank, world)
        srays9, srgbs_c = synthetic.train_rays(shi - slo, seed=7 + rank)
        srays_h, srgbs_h = srays9[:, :8].contiguous().pin_memory(), srgbs_c.contiguous().pin_memory()
        srays, srgbs = srays_h.to(dev), srgbs_h.to(dev)

        def static_step(rays_in=None, rgbs_in=None):
            r_in = srays if rays_in is None else rays_in
            t_in = srgbs if rgbs_in is None else rgbs_in
            for m in smodels:
                m.zero_grad(set_to_none=True)
            total = torch.zeros((), device=dev)
            sc = 16384    # rays per chunk: 128 + 256 samples per ray, ~50 GB of stashes alive per chunk
            for i in range(0, r_in.shape[0], sc):
                out = static_render_rays(smodels, semb, r_in[i:i + sc], N_samples=128, perturb=1.0, noise_std=1.0,
                                         N_importance=128)
                tgt = t_in[i:i + sc]
                loss = (torch.nn.functional.mse_loss(out['rgb_coarse'], tgt, reduction='sum') +
                        torch.nn.functional.mse_loss(out['rgb_fine'], tgt, reduction='sum')) / (3.0 * n_static)
                loss.backward()
                total += loss.detach()
            return total

        def static_e2e():
            loss = static_step(srays_h.to(dev, non_blocking=True), srgbs_h.to(dev, non_blocking=True))
            loss_h.copy_(loss, non_blocking=True)
            torch.cuda.current_stream().synchronize()

        static_step()
        ssteps = max(3, args.static_steps)
        secs_s, launches_s, prof_s = timed_loop(static_step, ssteps, profile=True)
        static_e2e()
        secs_se, _, _ = timed_loop(static_e2e, ssteps)
        sk, sexec = kernel_table(prof_s, secs_s, STATIC_FLOP_PER_EVAL, STATIC_FLOP_PER_EVAL)
        static = {"value": n_static * ssteps / secs_s, "unit": "rays/s", "rays_per_step": n_static, "samples": "128+128",
                  "ms_per_step": 1e3 * secs_s / ssteps, "steps_timed": ssteps,
                  "e2e": {"value": n_static * ssteps / secs_se, "unit": "rays/s",
                          "h2d_bytes_per_step": int(srays_h.numel() * 4 + srgbs_h.numel() * 4), "d2h_bytes_per_step": 4},
                  "gpu_launches": launches_s, "roofline": roofline_of(sk, sexec, secs_s, peaks, {}),
                  "workload": "cfg4: static NeRF baseline, 262144-ray batch, perturb=1, noise_std=1, fwd+bwd"}
        del smodels, srays, srgbs
        torch.cuda.empty_cache()

    # ---------------------------------------------------------------------------------------------------------------
    # secondary workload (BASELINE.json configs[4]): SE3Field warp + axis-aligned slicing (H = G = 8), 131 072-ray batch
    # sharded over the ranks, 128+128 samples, noise_std=1, forward + loss + backward + Adam, chunks of --chunk / 2 rays
    # ---------------------------------------------------------------------------------------------------------------
    se3 = None
    if not args.no_se3:
        n_se3 = 131072
        m5 = NerfModel(emb, **SE3_KW)
        m5.load_state_dict(synthetic.make_state_dict(m5, seed=0, boosted=False))
        m5 = m5.to(dev)
        fg5 = hn_train.FlatGrads(m5.parameters())
        m5.attach_flat_grads(fg5)
        opt5 = hn_train.FusedAdam(fg5, lr=5e-4, eps=1e-8)
        lo5, hi5 = hn_train.shard_bounds(n_se3, rank, world)
        r5, c5 = synthetic.train_rays(n_se3, seed=11)
        r5_h, c5_h = r5[lo5:hi5].contiguous().pin_memory(), c5[lo5:hi5].contiguous().pin_memory()
        r5_d, c5_d = r5_h.to(dev), c5_h.to(dev)

        def se3_step(rays_in=None, rgbs_in=None):
            return hn_train.train_step(m5, r5_d if rays_in is None else rays_in, c5_d if rgbs_in is None else rgbs_in, fg5,
                                       global_rays=n_se3, chunk=max(1024, args.chunk // 2), optimizer=opt5)

        g5 = None
        if use_graph:
            try:
                g5 = hn_train.GraphedTrainStep(m5, fg5, hi5 - lo5, n_se3, min(max(1024, args.chunk // 2), 4096))
                g5(r5_d, c5_d, opt5)
                torch.cuda.synchronize()
            except Exception:   # noqa: BLE001
                g5 = None
                torch.cuda.synchronize()

        def se3_e2e():
            r, c = r5_h.to(dev, non_blocking=True), c5_h.to(dev, non_blocking=True)
            loss = g5(r, c, opt5) if g5 is not None else se3_step(r, c)
            loss_h.copy_(loss, non_blocking=True)
            torch.cuda.current_stream().synchronize()

        se3_step()
        steps5 = max(3, args.se3_steps)
        secs_5, launches_5, prof_5 = timed_loop(se3_step, steps5, profile=True)
        se3_e2e()
        secs_5e, _, _ = timed_loop(se3_e2e, steps5)
        k5, exec5 = kernel_table(prof_5, secs_5, SE3_FLOP_PER_EVAL, SE3_TRUNK_FLOP_PER_EVAL)
        se3 = {"value": n_se3 * steps5 / secs_5, "unit": "rays/s", "rays_per_step": n_se3, "samples": "128+128",
               "ms_per_step": 1e3 * secs_5 / steps5, "steps_timed": steps5,
               "e2e": {"value": n_se3 * steps5 / secs_5e, "unit": "rays/s",
                       "h2d_bytes_per_step": int(r5_h.numel() * 4 + c5_h.numel() * 4), "d2h_bytes_per_step": 4},
               "gpu_launches": launches_5, "roofline": roofline_of(k5, exec5, secs_5, peaks, {}),
               "workload": "cfg5: SE3Field warp + axis-aligned slicing (hyper point = GLO vector, H = G = 8), 131072-ray batch, "
                           "128+128 samples, noise_std=1, fwd+loss+bwd+Adam; parity is against the batched restatement "
                           "(the reference never instantiates SE3Field)"}
        se3["e2e"]["launch"] = "CUDA graph" if g5 is not None else "eager"
        del m5, fg5, opt5, r5_d, c5_d, g5
        torch.cuda.empty_cache()

    print(f"[bench] rank {rank}: peak device memory reserved {torch.cuda.max_memory_reserved() / 2**30:.1f} GiB", file=sys.stderr)
    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            cpu = cpu_reference_rate(n_rays=1024, repeats=2, warmup=1, workload="train")
            if se3 is not None:
                se3["cpu_baseline"] = cpu_reference_rate(n_rays=256, repeats=1, warmup=1, workload="se3")
            if render is not None:
                render["cpu_baseline"] = cpu_reference_rate(n_rays=1024, repeats=2, warmup=1, workload="render")
            if static is not None:
                static["cpu_baseline"] = cpu_reference_rate(n_rays=512, repeats=1, warmup=1, workload="static")
        rays_per_s = GLOBAL_RAYS * args.steps / secs
        line = {
            "metric": METRIC, "value": rays_per_s, "unit": "rays/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": 1e3 * secs / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": WORKLOAD, "global_rays": GLOBAL_RAYS, "rays_per_gpu": hi - lo, "chunk_rays": chunk,
                       "samples": f"{N_COARSE}+{N_FINE}", "parallelism": f"dp{world} (ray shards, 1 flat NCCL all-reduce/step)",
                       "optimizer": "Adam step inside the timed region", "timing": "CUDA events per step, max over ranks",
                       "train_state": "every timed step starts from the initial weights and Adam state (restored between steps, "
                                      "outside the events)",
                       "l2": "256 MB buffer written between timed steps; per-step working set (>10 GB) exceeds L2",
                       "flop_accounting": "roofline.* count EXECUTED unpadded FLOPs (the fine level's 64 inherited depths skip "
                                          "the shared warp / sheet nets: 874.3 MFLOP per ray instead of the reference's 923.4)",
                       "dp_parity": dp_parity},
            "e2e": {"value": GLOBAL_RAYS * args.steps / secs_e2e, "unit": "rays/s",
                    "h2d_bytes_per_step": int(rays_h.numel() * 4 + rgbs_h.numel() * 4), "d2h_bytes_per_step": 4,
                    "launch": graph_note},
            "gpu_launches": launches, "clocks": clk, "roofline": roof, "cpu_baseline": cpu, "render": render, "static_nerf": static,
            "se3_axis": se3,
        }
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(out_dir, arrays):
    """Writes every tensor of `arrays` as float32 to out_dir/<name>.npy."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


_REAL_STDOUT = None


def emit(line):
    """The ONE JSON line of the contract goes to the process's real stdout; everything else any library prints on
    fd 1 during the run (e.g. NCCL's version banner at N > 1) has been redirected to stderr by main()."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--chunk", type=int, default=16384,
                    help="rays per forward/backward chunk on one GPU (64+64 samples: 1 M samples per launch, ~38 GB of "
                         "stashes alive per chunk; 8192 costs 1.5 %% of the step in launch gaps, 32768 gains another 1 %% "
                         "for twice the memory)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-render", action="store_true", help="skip the secondary full-frame render measurement")
    ap.add_argument("--no-static", action="store_true", help="skip the secondary static-NeRF (cfg4) measurement")
    ap.add_argument("--render-frames", type=int, default=5, help="timed frames of the render leg (>= 5)")
    ap.add_argument("--render-chunk", type=int, default=131072, help="rays per chunk of the render leg")
    ap.add_argument("--static-steps", type=int, default=3, help="timed steps of the static-NeRF leg (>= 3)")
    ap.add_argument("--no-se3", action="store_true", help="skip the secondary SE3 + axis-aligned (cfg5) measurement")
    ap.add_argument("--graph-chunk", type=int, default=16384, help="rays per chunk inside the CUDA graph of the end-to-end path")
    ap.add_argument("--no-graph", action="store_true", help="end-to-end path: launch the chunk loop eagerly instead of from a CUDA graph")
    ap.add_argument("--se3-steps", type=int, default=3, help="timed steps of the cfg5 leg (>= 3)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed train steps, write the last step's loss, gradient and updated parameters as "
                         "float32 DIR/<name>.npy (inputs and draws are seeded: same arguments, same inputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
