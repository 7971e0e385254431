"""Cost of the annealed positional encodings (extra_params alphas): the cfg2 train step (65 536 rays, 64 + 64 samples,
chunks of 8 192) and a cfg3 render (262 144 rays, 64 + 128 samples, no_grad), each alternated with windows off
(all alphas None: hn_pack_weights / hn_mlp_bwd_*weights) and on (fractional alphas: the *_windowed entry points), in one
process.  The forward and data-gradient kernels are the same in both modes; only the weight packing and the weight
gradient's flush differ, and their per-call times are printed on their own lines.

    python profiles/posenc_window_cost.py [--rounds 5] [--out posenc_window_cost.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from hypernerf_torch_b200 import _lib, _packing, synthetic  # noqa: E402
from hypernerf_torch_b200 import train as hn_train  # noqa: E402
from hypernerf_torch_b200.models import NerfModel  # noqa: E402

DEV = "cuda"
EMB = {'warp': list(range(100)), 'camera': [0], 'appearance': list(range(100)), 'time': list(range(100))}
ON = {'warp_alpha': 3.5, 'hyper_sheet_alpha': 2.25, 'nerf_alpha': 6.5, 'hyper_alpha': 1.5}


def cfg_kwargs(n_fine, noise_std):
    return dict(near=0., far=1., n_samples_coarse=64, n_samples_fine=n_fine, noise_std=noise_std,
                hyper_slice_method='bendy_sheet', hyper_slice_out_dim=2, use_warp=True, use_nerf_embed=False,
                use_alpha_cond=False, use_rgb_cond=False, GLO_dim=8, share_GLO=True, xyz_fourier_dim=10,
                hyper_fourier_dim=6, view_fourier_dim=6)


def device_info():
    info = {"device": torch.cuda.get_device_name()}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip().splitlines()[torch.cuda.current_device()]
    except Exception as e:   # the numbers still stand; the card's setting is then unknown
        info["power_limit_and_max_sm_clock"] = f"unavailable ({e})"
    return info


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
    ap.add_argument("--train-rays", type=int, default=65536)
    ap.add_argument("--render-rays", type=int, default=262144)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("posenc_window_cost.py measures on the GPU; there is no CPU fallback")
    torch.manual_seed(0)
    train_model = NerfModel(EMB, **cfg_kwargs(64, 1.0)).to(DEV)
    fg = hn_train.FlatGrads(train_model.parameters())
    train_model.attach_flat_grads(fg)
    rays, rgbs = synthetic.train_rays(args.train_rays, seed=1, device=DEV)
    render_model = NerfModel(EMB, **cfg_kwargs(128, None)).to(DEV)
    rrays, _ = synthetic.train_rays(args.render_rays, seed=2, device=DEV)

    modes = {"off": None, "on": ON}

    def train(mode):
        hn_train.train_step(train_model, rays, rgbs, fg, chunk=8192, extra_params=modes[mode])

    def render(mode):
        hn_train.render_rays(render_model, rrays, extra_params=modes[mode])

    for mode in modes:                          # warm-up of every shape and both plan tables
        train(mode)
        render(mode)
    res = {f"{w}_{m}": [] for w in ("train_ms", "render_ms") for m in modes}
    for _ in range(args.rounds):
        for mode in modes:
            res[f"train_ms_{mode}"].append(timed_ms(lambda: train(mode), 3))
            res[f"render_ms_{mode}"].append(timed_ms(lambda: render(mode), 2))

    # per-call kernel times: packing of both levels, and the weight-gradient launches of one train step
    pack = {}
    for mode in modes:
        win = _packing.pe_alphas(modes[mode])
        pack[mode] = timed_ms(lambda: train_model.refresh_packed(win), 50) / 2       # two levels per refresh
    wgrad = {}
    for mode in modes:
        _lib.profile = []
        train(mode)
        torch.cuda.synchronize()
        calls = [(n, e0.elapsed_time(e1)) for n, _, e0, e1 in _lib.profile if n.startswith("mlp_wgrad")]
        _lib.profile = None
        wgrad[mode] = {"calls": len(calls), "mean_ms": statistics.mean(t for _, t in calls)}

    out = device_info()
    out.update({k: {"median": statistics.median(v), "min": min(v), "max": max(v)} for k, v in res.items()})
    out["pack_kernel_ms_per_level"] = pack
    out["wgrad_ms_per_call"] = wgrad
    out["train_rays"], out["render_rays"], out["rounds"] = args.train_rays, args.render_rays, args.rounds
    print(f"device {out['device']}, power limit / max SM clock {out['power_limit_and_max_sm_clock']}")
    for w in ("train_ms", "render_ms"):
        print(f"{w}: off median {out[w + '_off']['median']:.2f} [{out[w + '_off']['min']:.2f}, {out[w + '_off']['max']:.2f}]"
              f"  on median {out[w + '_on']['median']:.2f} [{out[w + '_on']['min']:.2f}, {out[w + '_on']['max']:.2f}]")
    print(f"weight packing per level (refresh_packed: host call + pack_kernel): off {pack['off'] * 1e3:.1f} us  on {pack['on'] * 1e3:.1f} us")
    print(f"weight gradient per call: off {wgrad['off']['mean_ms'] * 1e3:.1f} us  on {wgrad['on']['mean_ms'] * 1e3:.1f} us"
          f"  ({wgrad['on']['calls']} calls per step)")
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
