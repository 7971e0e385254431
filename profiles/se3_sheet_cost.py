"""Cost of the SE3 warp with bendy-sheet slicing (H = 2, HyperNeRF's "DS" model) next to config 5 (SE3 warp +
axis-aligned slicing, H = 8), in one process: train-step rays/s at 131 072 rays and 128 + 128 samples (chunks of 8 192
rays, as bench.py's se3 leg), render Mrays/s (no_grad) on the same rays, per-1 M-sample times of the full network's
forward, data gradient and weight gradient inside the train step (CUDA events around every launch), and the algorithmic
MAC per sample evaluation from the modules' shapes.  The two models are alternated round by round.

    python profiles/se3_sheet_cost.py [--rounds 5] [--out se3_sheet_cost.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from hypernerf_torch_b200 import _lib, synthetic  # noqa: E402
from hypernerf_torch_b200 import train as hn_train  # noqa: E402
from hypernerf_torch_b200.models import NerfModel  # noqa: E402

DEV = "cuda"
EMB = {'warp': list(range(100)), 'camera': [0], 'appearance': list(range(100)), 'time': list(range(100))}
MODELS = {"se3_sheet_h2": dict(hyper_slice_method='bendy_sheet', hyper_slice_out_dim=2),
          "se3_axis_h8": dict(hyper_slice_method='axis_aligned_plane', hyper_slice_out_dim=8)}


def kwargs(conf, noise_std):
    kw = dict(near=0., far=1., n_samples_coarse=128, n_samples_fine=128, noise_std=noise_std, use_warp=True,
              use_nerf_embed=False, use_alpha_cond=False, use_rgb_cond=False, GLO_dim=8, share_GLO=True,
              xyz_fourier_dim=10, hyper_fourier_dim=6, view_fourier_dim=6, warp_field_type='se3')
    kw.update(MODELS[conf])
    return kw


def device_info():
    info = {"device": torch.cuda.get_device_name()}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip().splitlines()[torch.cuda.current_device()]
    except Exception as e:   # the numbers still stand; the card's setting is then unknown
        info["power_limit_and_max_sm_clock"] = f"unavailable ({e})"
    return info


def mac_per_sample(model):
    """Multiply-accumulates of one sample evaluation through the whole network: every nn.Linear of the warp field, the
    hyper sheet and one level's template (its in x out), unpadded."""
    subs = [model.warp_field, model.nerf_mlps_coarse] + ([model.hyper_sheet_mlp] if hasattr(model, "hyper_sheet_mlp") else [])
    return sum(m.in_features * m.out_features for s in subs for m in s.modules() if isinstance(m, torch.nn.Linear))


def timed_ms(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--rays", type=int, default=131072)
    ap.add_argument("--chunk", type=int, default=8192)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("se3_sheet_cost.py measures on the GPU; there is no CPU fallback")
    torch.manual_seed(0)
    rays, rgbs = synthetic.train_rays(args.rays, seed=11, device=DEV)
    train_m, render_m, fgs = {}, {}, {}
    for conf in MODELS:
        m = NerfModel(EMB, **kwargs(conf, 1.0))
        m.load_state_dict(synthetic.make_state_dict(m, seed=1))
        train_m[conf] = m.to(DEV)
        fgs[conf] = hn_train.FlatGrads(m.parameters())
        m.attach_flat_grads(fgs[conf])
        r = NerfModel(EMB, **kwargs(conf, None))
        r.load_state_dict(synthetic.make_state_dict(r, seed=1))
        render_m[conf] = r.to(DEV)

    def train(conf):
        hn_train.train_step(train_m[conf], rays, rgbs, fgs[conf], chunk=args.chunk)

    def render(conf):
        hn_train.render_rays(render_m[conf], rays, chunk=args.chunk)

    for conf in MODELS:          # warm-up of every shape
        train(conf)
        render(conf)
    res = {f"{w}_ms_{c}": [] for w in ("train", "render") for c in MODELS}
    for _ in range(args.rounds):
        for conf in MODELS:
            res[f"train_ms_{conf}"].append(timed_ms(lambda: train(conf), 2))
            res[f"render_ms_{conf}"].append(timed_ms(lambda: render(conf), 2))
    kernels = {}
    for conf in MODELS:          # per-launch CUDA events of one train step and one render
        kernels[conf] = {}
        for what, fn in (("train", train), ("render", render)):
            _lib.profile = []
            fn(conf)
            torch.cuda.synchronize()
            calls = _lib.profile
            _lib.profile = None
            for name in ("mlp_fwd", "mlp_dgrad", "mlp_wgrad"):
                sel = [(n, e0.elapsed_time(e1)) for k, n, e0, e1 in calls if k == name]
                if sel:
                    key = f"{name}{'_inference' if what == 'render' else ''}_ms_per_1M_samples"
                    kernels[conf][key] = sum(t for _, t in sel) / sum(n for n, _ in sel) * 1e6

    out = device_info()
    out["rays"], out["samples"], out["chunk"], out["rounds"] = args.rays, "128+128", args.chunk, args.rounds
    for conf in MODELS:
        tr, rr = statistics.median(res[f"train_ms_{conf}"]), statistics.median(res[f"render_ms_{conf}"])
        out[conf] = {"train_rays_per_s": args.rays / tr * 1e3,
                     "train_ms": {"median": tr, "min": min(res[f"train_ms_{conf}"]), "max": max(res[f"train_ms_{conf}"])},
                     "render_mrays_per_s": args.rays / rr * 1e-3,
                     "render_ms": {"median": rr, "min": min(res[f"render_ms_{conf}"]), "max": max(res[f"render_ms_{conf}"])},
                     "mac_per_sample": mac_per_sample(train_m[conf]), **kernels[conf]}
    print(f"device {out['device']}, power limit / max SM clock {out['power_limit_and_max_sm_clock']}")
    for conf in MODELS:
        o = out[conf]
        print(f"{conf}: train {o['train_rays_per_s'] / 1e3:.1f} k rays/s (median {o['train_ms']['median']:.1f} ms, "
              f"[{o['train_ms']['min']:.1f}, {o['train_ms']['max']:.1f}]), render {o['render_mrays_per_s']:.3f} Mrays/s, "
              f"{o['mac_per_sample']} MAC/sample")
        print("   per 1 M samples: " + ", ".join(f"{k.replace('_ms_per_1M_samples', '')} {v:.2f} ms"
                                               for k, v in o.items() if k.endswith("per_1M_samples")))
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
