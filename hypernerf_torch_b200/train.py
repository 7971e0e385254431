"""Train-step plumbing around the drop-in NerfModel: what NeRFSystem.training_step (train.py:147-163) + the
ShardedDDP gradient reduction (train.py:224-229) do, without Lightning.

* `FlatGrads` makes every parameter's `.grad` a view of one flat fp32 buffer, so the data-parallel exchange is ONE
  NCCL all-reduce of 5.9 MB per step (SURVEY.md §2.2 / §8(e)) and zeroing is one memset.
* `train_step` runs forward + MSE(coarse) + MSE(fine) (losses.py:9-14) + backward over the local ray shard in
  chunks of `chunk` rays (activation stash of the fused backward is ~8.6 KB per sample, so 65 536 rays do not fit
  in one piece), accumulating gradients; the loss is scaled so the accumulated gradient equals that of the mean
  over the GLOBAL batch, then all-reduced (sum) across ranks.
"""
import torch
import torch.distributed as dist

from . import _lib, _packing, losses, model_utils

EXTRA_PARAMS = {'nerf_alpha': None, 'warp_alpha': None, 'hyper_alpha': None, 'hyper_sheet_alpha': None}


class FlatGrads:
    def __init__(self, params):
        self.params = [p for p in params if p.requires_grad]
        total, self.offsets = 0, []
        for p in self.params:
            self.offsets.append(total)
            total += (p.numel() + 3) // 4 * 4
        p0 = self.params[0]
        self.flat = torch.zeros(total, device=p0.device, dtype=p0.dtype)
        self.bind()

    def offset_of(self, param):
        """Element offset of `param`'s gradient inside `flat` (KeyError if it is not one of this buffer's parameters)."""
        if getattr(self, "_by_id", None) is None:
            self._by_id = {id(p): off for p, off in zip(self.params, self.offsets)}
        return self._by_id[id(param)]

    def c_offsets(self):
        import ctypes
        if getattr(self, "_c_offs", None) is None:
            self._c_offs = (ctypes.c_int64 * len(self.offsets))(*self.offsets)
        return self._c_offs

    def bind(self):
        for p, off in zip(self.params, self.offsets):
            p.grad = self.flat[off:off + p.numel()].view_as(p)

    def zero(self):
        self.flat.zero_()
        for p, off in zip(self.params, self.offsets):
            if p.grad is None or p.grad.data_ptr() != self.flat.data_ptr() + 4 * off:
                self.bind()
                break

    def all_reduce(self):
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            dist.all_reduce(self.flat, op=dist.ReduceOp.SUM)


class FusedAdam:
    """torch.optim.Adam (utils/__init__.py:22-41: lr, eps=1e-8, weight_decay; betas (0.9, 0.999)) as ONE launch of
    hn_adam_step over flat buffers (SURVEY.md §8(f) row 1).

    The parameters of `flat_grads` are re-pointed into one flat fp32 buffer with the gradient buffer's offsets (the
    nn.Parameter objects, their names and state_dict stay what they were), exp_avg / exp_avg_sq are flat too.
    `param_groups[0]['lr']` is read every step, so torch.optim.lr_scheduler classes can drive it."""

    def __init__(self, flat_grads, lr=5e-4, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0):
        from . import _lib
        self._lib = _lib
        self.fg = flat_grads
        if flat_grads.flat.device.type != 'cuda':
            raise _lib.NativeLibraryError("FusedAdam needs CUDA parameters (no CPU path)")
        self.flat = torch.zeros_like(flat_grads.flat)
        with torch.no_grad():
            for p, off in zip(flat_grads.params, flat_grads.offsets):
                view = self.flat[off:off + p.numel()].view_as(p)
                view.copy_(p)
                p.data = view
        self.exp_avg = torch.zeros_like(self.flat)
        self.exp_avg_sq = torch.zeros_like(self.flat)
        self.step_count = 0
        self.defaults = dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay)
        self.param_groups = [dict(params=flat_grads.params, lr=lr, betas=betas, eps=eps, weight_decay=weight_decay,
                                  initial_lr=lr)]

    def zero_grad(self, set_to_none=False):
        self.fg.zero()

    @torch.no_grad()
    def step(self, grad_scale=1.0):
        L, g = self._lib, self.param_groups[0]
        self.step_count += 1
        L.check(L.lib().hn_adam_step(L.ptr(self.flat), L.ptr(self.fg.flat), L.ptr(self.exp_avg), L.ptr(self.exp_avg_sq),
                                     self.flat.numel(), g['lr'], g['betas'][0], g['betas'][1], g['eps'],
                                     g['weight_decay'], self.step_count, grad_scale, L.stream()), "hn_adam_step")
        L.count(1)
        # the parameters changed behind autograd's back: bump their version counters (the packed-weight cache of the
        # models keys on them)
        torch.autograd.graph.increment_version(self.fg.params)

    def state_dict(self):
        return dict(step=self.step_count, exp_avg=self.exp_avg, exp_avg_sq=self.exp_avg_sq,
                    param_groups=[{k: v for k, v in self.param_groups[0].items() if k != 'params'}])

    def load_state_dict(self, sd):
        self.step_count = int(sd['step'])
        self.exp_avg.copy_(sd['exp_avg'])
        self.exp_avg_sq.copy_(sd['exp_avg_sq'])
        self.param_groups[0].update(sd['param_groups'][0])


def shard_bounds(n, rank, world):
    """Contiguous split of n rays over `world` ranks (SURVEY.md §8(e))."""
    per = (n + world - 1) // world
    lo = min(rank * per, n)
    return lo, min(lo + per, n)


def _extra(extra_params):
    """EXTRA_PARAMS with the caller's entries on top."""
    return {**EXTRA_PARAMS, **(extra_params or {})}


def train_step(model, rays, rgbs, flat_grads, global_rays=None, chunk=8192, optimizer=None, return_stats=False,
               _exchange=True, extra_params=None, _window=None):
    """One data-parallel training step on this rank's ray rows (B,9) / target colours (B,3).
    Returns the local contribution to the global-mean loss (sum over ranks = the reference's loss); with
    return_stats, training_step's log entries {'train/loss', 'train/psnr'} (train.py:147-163; psnr of the fine level
    over this rank's rays, metrics.py:4-13) as device tensors.  extra_params: the forward's `extra_params`
    ({'nerf_alpha', 'warp_alpha', 'hyper_alpha', 'hyper_sheet_alpha'}: the coarse-to-fine encoding windows; unset = none)."""
    B = rays.shape[0]
    global_rays = B if global_rays is None else global_rays
    extra = _extra(extra_params)
    flat_grads.zero()
    total = torch.zeros((), device=rays.device, dtype=torch.float32)
    fine_sq = None
    # the weights do not change between the chunks of one step: pack the bf16 blobs once
    with model.packed_frozen(extra, _window=_window):
        for i in range(0, B, chunk):
            rows = rays[i:i + chunk]
            tgt = rgbs[i:i + chunk]
            out = model(model_utils.prepare_ray_dict(rows), dict(extra))
            # mean over the global batch: (sum_sq(coarse) + sum_sq(fine)) / (3 * global_rays), one fused kernel that
            # also seeds both levels' gradients (losses.py:9-14)
            loss, sums = losses.mse_coarse_fine(out, tgt, global_count=3.0 * global_rays)
            loss.backward()
            total += loss.detach()
            if return_stats:
                fine_sq = sums[1] if fine_sq is None else fine_sq + sums[1]
    if _exchange:
        flat_grads.all_reduce()
    if optimizer is not None:
        optimizer.step()
    if return_stats:
        return {'train/loss': total, 'train/psnr': -10.0 * torch.log10(fine_sq / (3.0 * B))}
    return total


class GraphedTrainStep:
    """`train_step` for a fixed per-rank batch shape with its per-chunk launches (zeroing, weight packing, both levels'
    forward / loss / backward: ~45 launches per 8 192-ray chunk) captured ONCE in a CUDA graph and replayed, so a step costs
    the host one graph launch + the gradient exchange + the optimizer launch.  That matters where a step is short (N = 8:
    11 ms) and the caller synchronises every step (the end-to-end path: rays in, loss out).  The random draws are made by
    the captured torch.rand / torch.randn calls (graph-safe Philox: every replay advances the generator), the exchange and
    the optimizer stay outside the graph (NCCL's own stream; Adam's lr / step number are launch arguments).

        step = GraphedTrainStep(model, flat_grads, n_rays, global_rays, chunk)
        loss = step(rays, rgbs, optimizer)          # first call captures; the result lives in a static buffer that the
                                                    # next call overwrites (a dict of such with return_stats=True)

    windowed=True captures the windowed weight packing / weight gradient (coarse-to-fine encoding windows) over a persistent
    4-float device buffer of alphas; `step(rays, rgbs, optimizer, extra_params)` writes it before the replay (no host
    synchronisation, no new capture), so a schedule changes the alphas every step.  Unset alphas mean no window."""

    def __init__(self, model, flat_grads, n_rays, global_rays=None, chunk=8192, return_stats=False, windowed=False):
        dev = flat_grads.flat.device
        self.model, self.fg = model, flat_grads
        self.global_rays = n_rays if global_rays is None else global_rays
        self.chunk, self.return_stats = chunk, return_stats
        self.rays = torch.zeros(n_rays, 9, device=dev, dtype=torch.float32)
        self.rgbs = torch.zeros(n_rays, 3, device=dev, dtype=torch.float32)
        self.windowed = windowed
        self.alphas = torch.full((4,), float('inf'), device=dev, dtype=torch.float32) if windowed else None
        self.graph, self.loss, self.launches = None, None, 0

    def _local(self):
        window = _packing._DeviceWindow(self.alphas) if self.windowed else None
        return train_step(self.model, self.rays, self.rgbs, self.fg, global_rays=self.global_rays, chunk=self.chunk,
                          return_stats=self.return_stats, _exchange=False, _window=window)

    def _capture(self):
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):           # warm-up off the capture: allocator pools, plan caches, kernel attributes
            for _ in range(2):
                self._local()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        before = _lib.launches
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            self.loss = self._local()
        self.graph, self.launches = graph, _lib.launches - before

    def __call__(self, rays, rgbs, optimizer=None, extra_params=None):
        window = _packing.pe_alphas(extra_params)
        if self.windowed:
            # from pinned memory: an asynchronous copy ordered before the replay (the caching host allocator keeps the
            # staging block alive until the copy has run)
            vals = window if window is not None else (float('inf'),) * 4
            self.alphas.copy_(torch.tensor(vals, dtype=torch.float32).pin_memory(), non_blocking=True)
        elif window is not None:
            raise ValueError("this GraphedTrainStep was captured without encoding windows: build it with windowed=True "
                             "to pass extra_params alphas")
        self.rays.copy_(rays, non_blocking=True)
        self.rgbs.copy_(rgbs, non_blocking=True)
        if self.graph is None:
            self._capture()
        self.graph.replay()
        _lib.count(self.launches)
        self.fg.all_reduce()
        if optimizer is not None:
            optimizer.step()
        return self.loss


class _Replay:
    """Replays a fixed list of tensors for the torch.rand / torch.randn calls of one forward (SURVEY.md App. A.5: the
    draws are made with the reference's own generator calls; data-parallel parity needs every rank to consume its slice of
    the SAME global draws, SURVEY.md §8(e))."""

    def __init__(self, tensors):
        self.tensors = list(tensors)

    def __enter__(self):
        self._rand, self._randn = torch.rand, torch.randn

        def take(*a, **k):
            return self.tensors.pop(0)

        torch.rand = torch.randn = take
        return self

    def __exit__(self, *exc):
        torch.rand, torch.randn = self._rand, self._randn


def global_draws(model, n_rays, device, seed):
    """The four draws of one forward over a batch of n_rays (rand[B,Nc], randn(B,Nc,1), rand(B,Nf), randn(B,Nc+Nf,1); the
    randn's only with noise) from one seeded generator."""
    g = torch.Generator(device=device).manual_seed(seed)
    Nc, Nf = model.num_coarse_samples, model.num_fine_samples
    noise = model.noise_std is not None and model.noise_std > 0
    out = [torch.rand(n_rays, Nc, device=device, generator=g)]
    if noise:
        out.append(torch.randn(n_rays, Nc, 1, device=device, generator=g))
    out.append(torch.rand(n_rays, Nf, device=device, generator=g))
    if noise:
        out.append(torch.randn(n_rays, Nc + Nf, 1, device=device, generator=g))
    return out


def dp_parity_check(model, flat_grads, rays, rgbs, seed=4321, tol=1e-4):
    """N-GPU step == 1-GPU step (SURVEY.md §4 / §8(e)): every rank runs train_step on its contiguous shard of (rays, rgbs)
    with its slice of globally drawn randoms and all-reduces; rank 0 also runs the whole batch alone; the all-reduced flat
    gradient must equal the single-rank one to `tol` (relative L2).  Returns the relative difference (same on all ranks).
    Leaves flat_grads zeroed."""
    world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
    rank = dist.get_rank() if world > 1 else 0
    n, dev = rays.shape[0], rays.device
    draws = global_draws(model, n, dev, seed)
    lo, hi = shard_bounds(n, rank, world)
    with _Replay([d[lo:hi] for d in draws]):
        train_step(model, rays[lo:hi], rgbs[lo:hi], flat_grads, global_rays=n, chunk=max(hi - lo, 1))
    sharded = flat_grads.flat.clone()
    rel = torch.zeros((), device=dev)
    if rank == 0:
        flat_grads.zero()
        with model.packed_frozen():
            with _Replay(list(draws)):
                out = model(model_utils.prepare_ray_dict(rays), dict(EXTRA_PARAMS))
            loss, _ = losses.mse_coarse_fine(out, rgbs, global_count=3.0 * n)
            loss.backward()
        rel = (sharded - flat_grads.flat).norm() / flat_grads.flat.norm()
    if world > 1:
        dist.broadcast(rel, src=0)
    flat_grads.zero()
    rel = float(rel)
    if not rel <= tol:
        raise AssertionError(f"data-parallel gradient differs from the single-GPU gradient: relative L2 {rel:.3e} > {tol}")
    return rel


def save_ckpt(model, path, epoch=0, global_step=0, optimizer=None, module_name='nerf'):
    """Checkpoint in the layout Lightning's ModelCheckpoint writes for NeRFSystem (train.py:71: the model is the
    attribute `nerf`, so its tensors are stored as `nerf.<name>` under 'state_dict'); readable by utils.load_ckpt
    (utils/__init__.py:66-88) of this package and of the reference."""
    blob = {'epoch': epoch, 'global_step': global_step,
            'state_dict': {f'{module_name}.{k}': v.detach().cpu().clone() for k, v in model.state_dict().items()}}
    if optimizer is not None:
        osd = optimizer.state_dict()
        blob['optimizer_states'] = [{k: (v.detach().cpu() if torch.is_tensor(v) else v) for k, v in osd.items()}]
    torch.save(blob, path)


def fit(model, rays, rgbs, num_epochs=1, batch_size=1024, lr=5e-4, weight_decay=0.0, decay_step=(20,), decay_gamma=0.1,
        chunk=8192, seed=0, ckpt_path=None, log_every=0, cuda_graph=False, extra_params=None):
    """Minimal stand-in for `Trainer.fit(NeRFSystem)` (train.py:35-233) on a ray pool that is already on the device:
    per epoch one shuffled pass over (rays (P,9), rgbs (P,3)) in batches of `batch_size` (train_dataloader,
    train.py:133-138: shuffle=True; the last short batch is kept, as DataLoader's drop_last=False does), each batch
    = train_step + Adam (get_optimizer, utils/__init__.py:22-41), MultiStepLR(decay_step, decay_gamma) stepped per epoch
    (get_scheduler 'steplr', utils/__init__.py:43-47; opt.py:62-75 defaults).  Under torch.distributed every rank
    passes its own shard of the pool (SURVEY.md §8(e)); gradients are all-reduced inside train_step.
    cuda_graph: replay the full-size batches from one CUDA graph (GraphedTrainStep); the last short batch of an epoch runs
    eagerly.  extra_params: the forward's encoding-window alphas (train_step), a dict or a callable step -> dict (a
    coarse-to-fine schedule; `step` counts from 0).  Returns a list of per-step dicts {'epoch', 'step', 'lr', 'train/loss',
    'train/psnr'} (training_step's log)."""
    distributed = dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
    fg = FlatGrads(model.parameters())
    model.attach_flat_grads(fg)
    opt = FusedAdam(fg, lr=lr, eps=1e-8, weight_decay=weight_decay)
    P = rays.shape[0]
    if distributed:
        # what DDP guarantees (train.py:224-229): every rank starts from rank 0's parameters, and every rank runs the
        # same number of steps — with unequal shards the ranks are cut to the shortest one, as DistributedSampler's
        # drop_last does, otherwise the all-reduce of the extra steps would never be matched
        dist.broadcast(opt.flat, src=0)
        model.invalidate_packed()
        n = torch.tensor([P], device=rays.device, dtype=torch.int64)
        dist.all_reduce(n, op=dist.ReduceOp.MIN)
        P = int(n.item())
    gen = torch.Generator(device=rays.device).manual_seed(seed)
    step, log = 0, []
    graphed = None
    for epoch in range(num_epochs):
        opt.param_groups[0]['lr'] = lr * decay_gamma ** sum(1 for m in decay_step if epoch >= m)
        order = torch.randperm(rays.shape[0], device=rays.device, generator=gen)[:P]
        for i in range(0, P, batch_size):
            idx = order[i:i + batch_size]
            r, t = rays[idx], rgbs[idx]
            # every rank holds P rows and the same batch boundaries, so the global batch is world * local
            world = dist.get_world_size() if distributed else 1
            extra = extra_params(step) if callable(extra_params) else extra_params
            if cuda_graph and r.shape[0] == batch_size:
                if graphed is None:
                    graphed = GraphedTrainStep(model, fg, batch_size, world * batch_size, chunk, return_stats=True,
                                               windowed=extra_params is not None)
                stats = {k: v.clone() for k, v in graphed(r, t, opt, extra).items()}
            else:
                stats = train_step(model, r, t, fg, global_rays=world * r.shape[0], chunk=chunk, optimizer=opt,
                                   return_stats=True, extra_params=extra)
            step += 1
            log.append({'epoch': epoch, 'step': step, 'lr': opt.param_groups[0]['lr'], **stats})
            if log_every and step % log_every == 0:
                print({k: (float(v) if torch.is_tensor(v) else v) for k, v in log[-1].items()})
        if ckpt_path is not None:
            save_ckpt(model, ckpt_path.format(epoch=epoch), epoch=epoch, global_step=step, optimizer=opt)
    return log


@torch.no_grad()
def render_rays(model, rays, chunk=32768, keys=('rgb', 'depth'), extra_params=None):
    """Chunked inference (eval.py:77-103 `batched_inference`), keeping only the per-ray outputs in `keys` of the
    fine level instead of concatenating every per-sample tensor (SURVEY.md §8(f) row 3).  extra_params: as in
    train_step."""
    outs = {k: [] for k in keys}
    extra = _extra(extra_params)
    with model.packed_frozen(extra):
        for i in range(0, rays.shape[0], chunk):
            out = model(model_utils.prepare_ray_dict(rays[i:i + chunk]), dict(extra))
            for k in keys:
                outs[k].append(out['fine'][k])
    return {k: torch.cat(v, 0) for k, v in outs.items()}
