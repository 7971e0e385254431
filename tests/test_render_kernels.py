"""GPU parity of the HBM-bound stages (sampling, resampling, compositing) against the oracle, through the C-ABI."""
import pytest
import torch

from helpers import orc
from hypernerf_torch_b200 import model_utils as mu
from hypernerf_torch_b200 import synthetic

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _rays(n, seed=0):
    rays, _ = synthetic.train_rays(n, seed=seed)
    rays = rays.to(DEV)
    return rays[:, :3].contiguous(), rays[:, 3:6].contiguous()


@pytest.mark.parametrize("B,Nc", [(1, 64), (37, 64), (1024, 64), (130, 128), (5, 33)])
def test_sample_along_rays_bit_exact(B, Nc):
    o, d = _rays(B)
    torch.manual_seed(5)
    z, pts = mu.sample_along_rays(o, d, Nc, 0., 1., True, False)
    torch.manual_seed(5)
    u = torch.rand([B, Nc], device=DEV)
    z_ref, pts_ref = orc.sample_along_rays(o, d, Nc, 0., 1., u)
    assert torch.equal(z, z_ref) and torch.equal(pts, pts_ref)
    z2, _ = mu.sample_along_rays(o, d, Nc, 0., 1., False, False)
    z2_ref, _ = orc.sample_along_rays(o, d, Nc, 0., 1., None)
    assert torch.equal(z2, z2_ref)


def _random_samples(B, S, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    sigma = torch.nn.functional.softplus(torch.randn(B, S, device=DEV, generator=g) * 2 + 1)
    rgb = torch.rand(B, S, 3, device=DEV, generator=g)
    z, _ = torch.sort(torch.rand(B, S, device=DEV, generator=g), -1)
    return sigma, rgb, z


@pytest.mark.parametrize("B,S", [(1, 64), (33, 64), (257, 128), (16, 192), (9, 256), (7, 50), (3, 384), (2, 1)])
@pytest.mark.parametrize("white,inf", [(False, True), (True, False)])
def test_composite_forward_and_backward(B, S, white, inf):
    o, d = _rays(B, seed=2)
    sigma, rgb, z = _random_samples(B, S, 11)
    sigma.requires_grad_(True); rgb.requires_grad_(True)
    out = mu.volumetric_rendering(rgb, sigma, z, d, white, sample_at_infinity=inf, _return_index=True)
    s2 = sigma.detach().clone().requires_grad_(True); r2 = rgb.detach().clone().requires_grad_(True)
    ref = orc.volumetric_rendering(r2, s2, z, d, white_bkgd=white, sample_at_infinity=inf)
    for k in ("rgb", "depth", "acc", "weights"):
        err = (out[k] - ref[k]).abs().max().item()
        assert err < 2e-5, (k, err)   # fp32 both sides; tolerance = scan-order rounding
    same = (out['_med_idx'] == ref['med_idx'])
    assert same.float().mean() >= 0.99 or B < 100
    assert (out['med_depth'][same] - ref['med_depth'][same]).abs().max() < 1e-6 if same.any() else True
    gen = torch.Generator(device=DEV).manual_seed(3)
    gr, gd, ga = (torch.randn(B, 3, device=DEV, generator=gen), torch.randn(B, device=DEV, generator=gen),
                  torch.randn(B, device=DEV, generator=gen))
    gw = torch.randn(B, S, device=DEV, generator=gen)
    loss = (out['rgb'] * gr).sum() + (out['depth'] * gd).sum() + (out['acc'] * ga).sum() + (out['weights'] * gw).sum()
    loss.backward()
    lref = (ref['rgb'] * gr).sum() + (ref['depth'] * gd).sum() + (ref['acc'] * ga).sum() + (ref['weights'] * gw).sum()
    lref.backward()
    for a, b, name in ((sigma.grad, s2.grad, "g_sigma"), (rgb.grad, r2.grad, "g_rgb")):
        err = (a - b).abs().max().item()
        scale = b.abs().max().item() + 1e-12
        assert err <= 2e-4 * scale + 1e-6, (name, err, scale)


def test_composite_rgb_only_gradient():
    B, S = 64, 128
    o, d = _rays(B, seed=4)
    sigma, rgb, z = _random_samples(B, S, 12)
    sigma.requires_grad_(True); rgb.requires_grad_(True)
    out = mu.volumetric_rendering(rgb, sigma, z, d, False)
    (out['rgb'] ** 2).sum().backward()
    s2 = sigma.detach().clone().requires_grad_(True); r2 = rgb.detach().clone().requires_grad_(True)
    (orc.volumetric_rendering(r2, s2, z, d)['rgb'] ** 2).sum().backward()
    assert (sigma.grad - s2.grad).abs().max() <= 2e-4 * s2.grad.abs().max() + 1e-7
    assert (rgb.grad - r2.grad).abs().max() <= 2e-4 * r2.grad.abs().max() + 1e-7


@pytest.mark.parametrize("B,Nc,Nf", [(1, 64, 64), (37, 64, 64), (512, 64, 128), (19, 128, 128), (9, 128, 64), (4, 16, 5),
                                     (3, 200, 300)])
def test_sample_pdf_bit_exact(B, Nc, Nf):
    o, d = _rays(B, seed=6)
    g = torch.Generator(device=DEV).manual_seed(Nc + Nf)
    z, _ = torch.sort(torch.rand(B, Nc, device=DEV, generator=g), -1)
    w = torch.rand(B, Nc, device=DEV, generator=g) ** 4
    w[:, Nc // 2:Nc // 2 + 3] = 0.0                      # empty bins -> denom < eps branch
    if B > 2:
        w[1] = 0.0                                          # all-zero ray
        w[2, 5] = 50.0                                      # one dominant bin
    u = torch.rand(B, Nf, device=DEV, generator=g)
    u[0, 0] = 0.0
    z_f, pts, inds = mu.sample_pdf_fused(z, w, o, d, Nf, u=u, want_inds=True)
    bins = .5 * (z[..., 1:] + z[..., :-1])
    z_ref, pts_ref, inds_ref = orc.sample_pdf(bins, w[..., 1:-1], o, d, z, u)
    assert torch.equal(inds.long(), inds_ref), "searchsorted bin indices must be bit-exact"
    assert torch.equal(z_f, z_ref), "sorted sample depths must be bit-exact"
    assert torch.equal(pts, pts_ref)
    assert (z_f[:, 1:] >= z_f[:, :-1]).all()
    # generic entry point with caller-provided bins / strided weights view (the reference call shape)
    torch.manual_seed(1)
    z_g, pts_g = mu.sample_pdf(bins, w[..., 1:-1], o, d, z, Nf, True)
    torch.manual_seed(1)
    u2 = torch.rand(B, Nf, device=DEV)
    z_ref2, _, _ = orc.sample_pdf(bins, w[..., 1:-1], o, d, z, u2)
    assert torch.equal(z_g, z_ref2)


@pytest.mark.parametrize("B,Nc,Nf", [(37, 64, 64), (130, 64, 128), (9, 128, 64), (19, 128, 128), (5, 96, 40)])
@pytest.mark.parametrize("case", ["random", "sorted_u", "unsorted_coarse", "ties", "peaked", "crowded_u", "edge_u"])
def test_sample_pdf_rank_tables(B, Nc, Nf, case):
    """hn_sample_pdf_ranks: where the merge put every coarse depth / the i-th smallest new sample (consumed as they are by
    hn_mlp_fwd / hn_mlp_fwd_trunk).  Fast kernel (64 / 128 shapes: ranks from the CDF bins + bit mask; its generic-merge
    branch for non-ascending coarse depths) and generic kernel (96 + 40) against the oracle's merge; the tie rule is the
    reference's stable torch.sort of cat([z_vals, z_samples]) (model_utils.py:227): coarse depths first."""
    o, d = _rays(B, seed=3)
    g = torch.Generator(device=DEV).manual_seed(Nc * 7 + Nf)
    z, _ = torch.sort(torch.rand(B, Nc, device=DEV, generator=g), -1)
    w = torch.rand(B, Nc, device=DEV, generator=g)
    u = torch.rand(B, Nf, device=DEV, generator=g)
    if case == "sorted_u":
        u = torch.linspace(0., 1. - torch.finfo(torch.float32).eps, Nf, device=DEV).expand(B, Nf).contiguous()
    elif case == "unsorted_coarse":
        z = z[:, torch.randperm(Nc, device=DEV, generator=g)].contiguous()
    elif case == "ties":
        w[:, 3:-3] = 0.0          # many new samples collapse onto bin edges; duplicates among the draws
        u[:, 1::2] = u[:, 0::2][:, :u[:, 1::2].shape[1]]
    elif case == "peaked":
        w = w ** 8                # a trained model's distribution: most samples in a handful of bins
    elif case == "crowded_u":     # draws that are not uniform: the fast kernel's bucket sort hands the ray to its bitonic network
        u = 0.5 + 0.01 * u
        u[1::2] = torch.rand(u[1::2].shape, device=DEV, generator=g) ** 6      # skewed: some buckets crowded, some rays not
    elif case == "edge_u":        # first / last bucket: 0, the largest float below 1, and a few equal draws
        u[:, 0] = 0.0
        u[:, 1] = 1.0 - 2.0 ** -24
        u[:, 2] = u[:, 1]
        u[:, 3] = 2.0 ** -30
    z_f, pts, inds, (pos_c, pos_n) = mu.sample_pdf_fused(z, w, o, d, Nf, u=u, want_inds=True, want_ranks=True)
    bins = .5 * (z[..., 1:] + z[..., :-1])
    z_ref, pts_ref, inds_ref = orc.sample_pdf(bins, w[..., 1:-1], o, d, z, u)
    assert torch.equal(z_f, z_ref) and torch.equal(pts, pts_ref) and torch.equal(inds.long(), inds_ref)
    pc, pn = pos_c.long(), pos_n.long()
    both = torch.cat([pc, pn], -1)
    assert torch.equal(torch.sort(both, -1).values, torch.arange(Nc + Nf, device=DEV).expand(B, -1)), "not a permutation"
    zs = torch.sort(z, -1).values
    assert torch.equal(torch.gather(z_f, 1, pc), zs)                       # coarse depth i sits at pos_c[i]
    assert (pc[:, 1:] > pc[:, :-1]).all() and (pn[:, 1:] > pn[:, :-1]).all()   # both tables ascending
    new_sorted = torch.gather(z_f, 1, pn)                                 # the new samples, ascending
    assert (new_sorted[:, 1:] >= new_sorted[:, :-1]).all()
    # tie rule: a coarse depth precedes the new samples equal to it  <=>  #(new < coarse_i) == pos_c[i] - i
    cnt = (new_sorted[:, None, :] < zs[:, :, None]).sum(-1)
    assert torch.equal(cnt, pc - torch.arange(Nc, device=DEV))


@pytest.mark.parametrize("case", ["sorted_u", "unsorted_coarse", "ties"])
def test_sample_pdf_merge_paths_bit_exact(case):
    """The kernel sorts only the new samples and merges them with the coarse depths; deterministic (ascending) draws skip
    the sort, non-ascending coarse depths are sorted first, ties between a coarse depth and a sample keep both."""
    B, Nc, Nf = 33, 64, 128
    o, d = _rays(B, seed=16)
    g = torch.Generator(device=DEV).manual_seed(99)
    z, _ = torch.sort(torch.rand(B, Nc, device=DEV, generator=g), -1)
    w = torch.rand(B, Nc, device=DEV, generator=g)
    u = torch.rand(B, Nf, device=DEV, generator=g)
    if case == "sorted_u":     # eval path: u = linspace(0, 1 - eps, Nf) for every ray (model_utils.py:188-190)
        u = torch.linspace(0., 1. - torch.finfo(torch.float32).eps, Nf, device=DEV).expand(B, Nf).contiguous()
    elif case == "unsorted_coarse":
        z = z[:, torch.randperm(Nc, device=DEV, generator=g)].contiguous()
    else:                      # coarse depths on a coarse grid and zero-width bins make samples coincide with depths
        z = (torch.round(z * 16) / 16).contiguous()
        u[:, ::3] = u[:, 1::3][:, :u[:, ::3].shape[1]]
    z_f, pts, inds = mu.sample_pdf_fused(z, w, o, d, Nf, u=u, want_inds=True)
    bins = .5 * (z[..., 1:] + z[..., :-1])
    z_ref, pts_ref, inds_ref = orc.sample_pdf(bins, w[..., 1:-1], o, d, z, u)
    assert torch.equal(inds.long(), inds_ref)
    assert torch.equal(z_f, z_ref)
    assert torch.equal(pts, pts_ref)


def test_sample_pdf_against_unmodified_reference_golden():
    """tests/golden/sample_pdf_ref.pt was produced by the UNMODIFIED reference function (hypernerf/model_utils.py:160-232,
    run on the CPU by tests/test_sample_pdf_reference.py) at 64+64 and 64+128.  The kernel must (a) be bit-exact with the
    oracle contract and (b) differ from the reference's own indices only where the draw lies within 4 ulp of a CDF edge
    (SURVEY.md App. A.4 (ii)); elsewhere the sorted depths agree up to the CDF-ulp / denom amplification."""
    from conftest import load_golden
    for case in load_golden("sample_pdf_ref"):
        Nc, Nf = case['Nc'], case['Nf']
        z, w, u = case['z'].to(DEV), case['weights'].to(DEV), case['u'].to(DEV)
        B = z.shape[0]
        o = torch.zeros(B, 3, device=DEV)
        d = torch.tensor([[0., 0., 2.]], device=DEV).expand(B, 3).contiguous()
        z_f, _, inds = mu.sample_pdf_fused(z, w, o, d, Nf, u=u, want_inds=True)
        bins = .5 * (z[..., 1:] + z[..., :-1])
        z_orc, _, inds_orc = orc.sample_pdf(bins, w[..., 1:-1], o, d, z, u)
        assert torch.equal(inds.long(), inds_orc) and torch.equal(z_f, z_orc)          # (a)
        ref_i, ref_cdf = case['ref_inds'].to(DEV).long(), case['ref_cdf'].to(DEV)
        mism = inds.long() != ref_i
        if mism.any():                                                                   # (b)
            rows, cols = torch.nonzero(mism, as_tuple=True)
            lo, hi = torch.minimum(inds.long(), ref_i)[rows, cols], torch.maximum(inds.long(), ref_i)[rows, cols]
            assert int((hi - lo).max()) == 1
            uu = u[rows, cols].double()
            ulp = torch.tensor(2.0 ** -24, device=DEV, dtype=torch.float64) * torch.pow(2.0, torch.floor(torch.log2(uu)) + 1)
            assert float(((uu - ref_cdf[rows, lo].double()).abs() / ulp).max()) <= 4.0
        assert int(mism.sum()) <= max(1, int(2e-5 * mism.numel()))
        clean = ~mism.any(-1)
        ref_sorted, _ = torch.sort(torch.cat([z, case['ref_samples'].to(DEV)], -1), -1)
        dz = (z_f - ref_sorted).abs()[clean]
        # (bit-exact with the oracle (a); the oracle-vs-reference depth bound is asserted in tests/test_sample_pdf_reference.py)
        assert float(dz.max()) <= 2e-2 and float((dz == 0).float().mean()) > 0.7


def test_sample_pdf_full_size_properties():
    """BASELINE cfg-2 size (65 536 rays): sortedness, coarse depths preserved, samples inside the bin range."""
    B, Nc, Nf = 65536, 64, 64
    o, d = _rays(B, seed=8)
    g = torch.Generator(device=DEV).manual_seed(0)
    z, _ = torch.sort(torch.rand(B, Nc, device=DEV, generator=g), -1)
    w = torch.rand(B, Nc, device=DEV, generator=g)
    z_f, pts = mu.sample_pdf_fused(z, w, o, d, Nf)
    assert (z_f[:, 1:] >= z_f[:, :-1]).all()
    bins = .5 * (z[..., 1:] + z[..., :-1])
    assert (z_f >= z[:, :1]).all() and (z_f <= z[:, -1:]).all()
    cnt = (z_f[:, :, None] == z[:, None, :]).any(1).all(-1)  # every coarse depth appears in the output
    assert cnt.all()
    assert (bins.min(-1).values <= z_f.max(-1).values).all()


@pytest.mark.parametrize("B", [1, 37, 8192, 70001])
def test_fused_mse_loss_matches_reference_formula(B):
    """losses.py:9-14 + metrics.py:4-13 through hn_mse_loss: loss, gradient seeds and PSNR."""
    from hypernerf_torch_b200 import losses, metrics
    g = torch.Generator(device=DEV).manual_seed(B)
    c = torch.rand(B, 3, device=DEV, generator=g, requires_grad=True)
    f = torch.rand(B, 3, device=DEV, generator=g, requires_grad=True)
    t = torch.rand(B, 3, device=DEV, generator=g)
    loss, sums = losses.mse_coarse_fine({'coarse': {'rgb': c}, 'fine': {'rgb': f}}, t)
    (3.0 * loss).backward()
    c2, f2 = c.detach().clone().requires_grad_(True), f.detach().clone().requires_grad_(True)
    ref = torch.nn.functional.mse_loss(c2, t) + torch.nn.functional.mse_loss(f2, t)
    (3.0 * ref).backward()
    assert abs(loss.item() - ref.item()) < 1e-5 * max(1.0, abs(ref.item()))
    assert torch.allclose(c.grad, c2.grad, rtol=1e-5, atol=1e-9) and torch.allclose(f.grad, f2.grad, rtol=1e-5, atol=1e-9)
    psnr = metrics.psnr_from_sum(sums[1], 3 * B)
    assert abs(psnr.item() - metrics.psnr(f.detach(), t).item()) < 1e-3
    only_coarse = losses.MSELoss()({'coarse': {'rgb': c.detach()}}, t)
    assert abs(only_coarse.item() - torch.nn.functional.mse_loss(c.detach(), t).item()) < 1e-6


def test_device_ray_generation_matches_reference_golden():
    """datasets/ray_utils.py:5-93 on the device (hn_make_ndc_rays) against rows generated by the reference's functions."""
    from conftest import load_golden
    from hypernerf_torch_b200 import ray_utils
    for case in load_golden("ndc_rays"):
        rays = ray_utils.frame_rays_ndc(case['H'], case['W'], case['focal'], case['c2w'], near_plane=1.0)
        ref = case['rays']
        assert rays.shape == ref.shape
        err = (rays.cpu() - ref).abs().max().item()
        print(f"ndc rays {case['H']}x{case['W']} max_abs_err {err:.2e}")
        assert err < 2e-5            # fp32, different association of the same formula
        with_id = ray_utils.frame_rays_ndc(case['H'], case['W'], case['focal'], case['c2w'], near_plane=1.0, image_id=7)
        assert with_id.shape[1] == 9 and torch.equal(with_id[:, :8], rays) and (with_id[:, 8] == 7).all()


@pytest.mark.parametrize("weight_decay", [0.0, 1e-2])
def test_fused_adam_matches_torch_adam(weight_decay):
    """hn_adam_step over the flat buffers == torch.optim.Adam(lr, eps=1e-8, weight_decay) (utils/__init__.py:22-41) on
    the cfg-1 parameter shapes, 12 steps of random gradients, with an lr change in between (scheduler behaviour)."""
    from hypernerf_torch_b200 import train as hn_train
    shapes = synthetic.cfg1_state_dict_shapes()
    sd = synthetic.make_state_dict(shapes, seed=0)
    mine = [torch.nn.Parameter(v.clone().cuda()) for v in sd.values()]
    ref = [torch.nn.Parameter(v.clone().cuda()) for v in sd.values()]
    fg = hn_train.FlatGrads(mine)
    opt = hn_train.FusedAdam(fg, lr=5e-4, eps=1e-8, weight_decay=weight_decay)
    topt = torch.optim.Adam(ref, lr=5e-4, eps=1e-8, weight_decay=weight_decay)
    g = torch.Generator(device="cuda").manual_seed(0)
    for it in range(12):
        if it == 6:
            opt.param_groups[0]['lr'] = 5e-5
            topt.param_groups[0]['lr'] = 5e-5
        fg.zero()
        for p, q in zip(mine, ref):
            grad = torch.randn(p.shape, device="cuda", generator=g) * 10.0 ** float(it % 4 - 3)
            p.grad.copy_(grad)          # view of the flat buffer
            q.grad = grad.clone()
        v0 = mine[0]._version
        opt.step()
        topt.step()
        assert mine[0]._version > v0    # packed-weight caches key on the version counter
    for name, p, q in zip(sd, mine, ref):
        assert p.data_ptr() >= opt.flat.data_ptr() and p.data_ptr() < opt.flat.data_ptr() + 4 * opt.flat.numel()
        torch.testing.assert_close(p.detach(), q.detach(), rtol=2e-6, atol=2e-8, msg=name)
    # padding between tensors stays untouched
    assert torch.isfinite(opt.flat).all()
