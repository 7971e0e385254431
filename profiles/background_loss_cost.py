"""Cost of the background regularisation.

  * The warp stage alone (hn_mlp_fwd_warp + hn_mlp_bwd_warp_*, what `apply_warp` / `map_points` / the background loss
    run) against the earlier route of `apply_warp` through the whole level-0 network (hn_mlp_fwd + hn_mlp_bwd with zero
    view directions and zero sigma / rgb gradients), forward + backward per 1 M points, with the flat gradient attached.
  * The cfg2 train step (65 536 rays, 64 + 64 samples, chunks of 8 192) without and with 16 384 background points.

Both alternate their two variants in one process; the GPU name and power limit are read in the same call.

    python profiles/background_loss_cost.py [--rounds 5] [--out background_loss_cost.json]
"""
import argparse
import json
import os
import statistics
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from hypernerf_torch_b200 import synthetic  # noqa: E402
from hypernerf_torch_b200 import train as hn_train  # noqa: E402
from hypernerf_torch_b200.models import NerfModel, _FusedMlp, _FusedWarp  # noqa: E402
from posenc_window_cost import EMB, cfg_kwargs, device_info, timed_ms  # noqa: E402

DEV = "cuda"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--points", type=int, default=1 << 20)
    ap.add_argument("--train-rays", type=int, default=65536)
    ap.add_argument("--background", type=int, default=16384)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("background_loss_cost.py measures on the GPU; there is no CPU fallback")
    torch.manual_seed(0)
    model = NerfModel(EMB, **cfg_kwargs(64, 1.0)).to(DEV)
    model.load_state_dict(synthetic.make_state_dict(model, seed=0))
    fg = hn_train.FlatGrads(model.parameters())
    model.attach_flat_grads(fg)

    # ---- warp stage alone vs the whole level-0 network, forward + backward
    B, S = args.points // 256, 256
    g = torch.Generator(device=DEV).manual_seed(1)
    pts = (torch.rand(B, S, 3, device=DEV, generator=g) * 2 - 1).contiguous()
    ids = torch.randint(0, 100, (B,), device=DEV, generator=g)
    gw = torch.randn(B, S, 5, device=DEV, generator=g)
    zero_dirs = torch.zeros(B, 3, device=DEV)

    def warp_only():
        warped = _FusedWarp.apply(model, None, pts, ids, *model._warp_params())
        torch.autograd.backward(warped, gw)

    def full_network():
        _, _, warped = _FusedMlp.apply(model, (0, None), pts, zero_dirs, ids, None, 0.0, *model._canonical_params())
        torch.autograd.backward(warped, gw)

    # ---- the train step with and without background points
    rays, rgbs = synthetic.train_rays(args.train_rays, seed=2, device=DEV)
    bg = (torch.rand(args.background, 3, device=DEV, generator=g) * 2 - 1).contiguous()

    def step(with_bg):
        hn_train.train_step(model, rays, rgbs, fg, chunk=8192, background_points=bg if with_bg else None)

    variants = {"warp_only": warp_only, "full_network": full_network,
                "step_without_bg": lambda: step(False), "step_with_bg": lambda: step(True)}
    with model.packed_frozen():
        warp_only()
        full_network()
    step(False)
    step(True)
    res = {k: [] for k in variants}
    for _ in range(args.rounds):
        with model.packed_frozen():
            res["warp_only"].append(timed_ms(warp_only, 5) * (1 << 20) / (B * S))
            res["full_network"].append(timed_ms(full_network, 5) * (1 << 20) / (B * S))
        res["step_without_bg"].append(timed_ms(lambda: step(False), 3))
        res["step_with_bg"].append(timed_ms(lambda: step(True), 3))

    out = device_info()
    out.update({k: {"median": statistics.median(v), "min": min(v), "max": max(v)} for k, v in res.items()})
    out.update(points=B * S, train_rays=args.train_rays, background=args.background, rounds=args.rounds)
    print(f"device {out['device']}, power limit / max SM clock {out['power_limit_and_max_sm_clock']}")
    for k in variants:
        unit = "ms per 1 M points (fwd + bwd)" if k in ("warp_only", "full_network") else "ms per step"
        print(f"{k:16s} median {out[k]['median']:.3f} [{out[k]['min']:.3f}, {out[k]['max']:.3f}] {unit}")
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
