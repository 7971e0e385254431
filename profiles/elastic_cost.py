"""Cost of the warp Jacobians and the elastic loss (translation warp, bendy sheet H = 2).

  * Per launch, CUDA events over many launches, per 1 M points: the warp-only primal forward with its stash
    (hn_mlp_fwd_warp), the tangent forward of the 3 input directions (hn_mlp_fwd_warp_tangent), the elastic loss
    (hn_elastic_loss), and the 3 data-gradient and 3 weight-gradient launches of the tangent backward.  The tangent
    forward is also reported against its MAC floor: 3 x 127 872 MAC per point at the dense BF16 data-sheet rate.
  * The bench workload's train step (65 536 rays, 64 + 64 samples, chunks of 8 192) with elastic_weight 0 and 0.01,
    alternated in one process on the same seeded rays.

The GPU name and power limit are read in the same call.

    python profiles/elastic_cost.py [--rounds 5] [--out elastic_cost.json]
"""
import argparse
import ctypes as C
import json
import os
import statistics
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from hypernerf_torch_b200 import _lib, synthetic  # noqa: E402
from hypernerf_torch_b200 import train as hn_train  # noqa: E402
from hypernerf_torch_b200._lib import check, lib, ptr, stream  # noqa: E402
from hypernerf_torch_b200.models import NerfModel, _JACOBIAN_NO_GRAD_SLOTS  # noqa: E402
from posenc_window_cost import EMB, cfg_kwargs, device_info  # noqa: E402

DEV = "cuda"
WARP_MAC = 127872            # MAC per point of the translation warp stage (cfg 1): 3 tangent planes do 3 x this
BF16_DENSE_FLOPS = 2.25e15   # NVIDIA HGX B200 data sheet, one GPU, dense BF16, 1 000 W


def events_ms(fn, iters):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(iters):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--points", type=int, default=1 << 20)
    ap.add_argument("--train-rays", type=int, default=65536)
    ap.add_argument("--elastic-weight", type=float, default=0.01)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("elastic_cost.py measures on the GPU; there is no CPU fallback")
    torch.manual_seed(0)
    model = NerfModel(EMB, **cfg_kwargs(64, 1.0)).to(DEV)
    model.load_state_dict(synthetic.make_state_dict(model, seed=0, boosted=True))
    fg = hn_train.FlatGrads(model.parameters())
    model.attach_flat_grads(fg)

    # ---- the launches of one Jacobian forward + elastic loss + tangent backward on B x S points
    B, S = args.points // 256, 256
    n = B * S
    g = torch.Generator(device=DEV).manual_seed(1)
    pts = (torch.rand(B, S, 3, device=DEV, generator=g) * 2 - 1).contiguous()
    ids = torch.randint(0, 100, (B,), device=DEV, generator=g)
    w = torch.rand(n, device=DEV, generator=g)
    d, L = C.byref(model._desc), lib()
    sizes = model._sizes(n)
    saved = torch.empty(sizes.warp_saved_bytes, device=DEV, dtype=torch.uint8)
    tangent = torch.empty(3 * sizes.warp_saved_bytes, device=DEV, dtype=torch.uint8)
    work = torch.empty(sizes.warp_workspace_bytes, device=DEV, dtype=torch.uint8)
    warped = torch.empty(B, S, 3 + model._desc.hyper_dim, device=DEV)
    jac = torch.empty(B, S, 3, 3, device=DEV)
    planes = torch.empty(3, n, 3 + model._desc.hyper_dim, device=DEV)
    sums = torch.zeros(1, device=DEV)
    scratch = torch.zeros(model._desc.num_embeddings * model._desc.glo_dim, device=DEV)
    scratch_offs = (C.c_int64 * _lib.HN_NUM_PARAM_TENSORS)(*([0] + [-1] * (_lib.HN_NUM_PARAM_TENSORS - 1)))
    w_offs = (C.c_int64 * _lib.HN_NUM_PARAM_TENSORS)(*model._flat_offsets())
    for slot in _JACOBIAN_NO_GRAD_SLOTS:
        w_offs[slot] = -1

    def primal():
        check(L.hn_mlp_fwd_warp(d, ptr(packed), ptr(pts), ptr(ids), B, S, ptr(warped), ptr(saved), None, stream()), "fwd_warp")

    def tangent_fwd():
        check(L.hn_mlp_fwd_warp_tangent(d, ptr(packed), ptr(pts), ptr(saved), B, S, ptr(jac), ptr(tangent), stream()),
              "fwd_warp_tangent")

    def loss():
        check(L.hn_elastic_loss(ptr(jac), ptr(w), n, -2.0, 0.03, 1e-6, 1.0, ptr(sums), ptr(planes),
                                model._desc.hyper_dim, stream()), "elastic_loss")

    def data3():
        for c in range(3):
            check(L.hn_mlp_bwd_warp_data(d, ptr(packed), ptr(ids), ptr(saved), ptr(planes[c]), B, S, scratch_offs,
                                         ptr(scratch), ptr(work), None, None, stream()), "bwd_warp_data")

    def weights3():
        for c in range(3):
            check(L.hn_mlp_bwd_warp_weights(d, tangent.data_ptr() + c * sizes.warp_saved_bytes, B, S, w_offs, ptr(fg.flat),
                                            ptr(work), None, stream()), "bwd_warp_weights")

    # ---- the train step with and without the elastic term
    rays, rgbs = synthetic.train_rays(args.train_rays, seed=2, device=DEV)

    def step(ew):
        torch.manual_seed(3)
        hn_train.train_step(model, rays, rgbs, fg, chunk=8192, elastic_weight=ew)

    launches = {"primal_fwd": primal, "tangent_fwd": tangent_fwd, "elastic_loss": loss, "data_grad_x3": data3,
                "weight_grad_x3": weights3}
    with model.packed_frozen():
        packed = model._packed_window(0, None)[0]
        for fn in launches.values():
            fn()
        torch.cuda.synchronize()
    step(0.0)
    step(args.elastic_weight)
    res = {k: [] for k in list(launches) + ["step_elastic_off", "step_elastic_on"]}
    for _ in range(args.rounds):
        with model.packed_frozen():
            packed = model._packed_window(0, None)[0]
            for k, fn in launches.items():
                res[k].append(events_ms(fn, 10) * (1 << 20) / n)
        for k, ew in (("step_elastic_off", 0.0), ("step_elastic_on", args.elastic_weight)):
            res[k].append(events_ms(lambda: step(ew), 3))

    out = device_info()
    out.update({k: {"median": statistics.median(v), "min": min(v), "max": max(v)} for k, v in res.items()})
    floor_ms = 3 * WARP_MAC * 2 * (1 << 20) / BF16_DENSE_FLOPS * 1e3
    out["tangent_fwd_mac_floor_ms_per_1M"] = floor_ms
    out.update(points=n, train_rays=args.train_rays, elastic_weight=args.elastic_weight, rounds=args.rounds)
    print(f"device {out['device']}, power limit / max SM clock {out['power_limit_and_max_sm_clock']}")
    for k in res:
        unit = "ms per step" if k.startswith("step") else "ms per 1 M points"
        print(f"{k:18s} median {out[k]['median']:.3f} [{out[k]['min']:.3f}, {out[k]['max']:.3f}] {unit}")
    print(f"tangent forward MAC floor (dense BF16 data-sheet rate) {floor_ms:.3f} ms per 1 M points = "
          f"{floor_ms / out['tangent_fwd']['median']:.1%} of the measured time")
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
