"""GPU (-m gpu): the raw-parameter entry (SURVEY.md section 8(f) row 1) -- render() over a GaussianModel stand-in
with the activations and the SH concatenation fused into the kernels -- against the getter path (torch exp / sigmoid /
F.normalize / cat + autograd through them) and against the compiled reference rasterizer under the same torch prologue."""
import pytest
import torch

import helpers
from raw_model import RawModel, Pipe, PipeUnfused

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
CHAIN = {"scaling", "scaling_t", "rotation", "rotation_r", "t"}


def _render_and_backward(model, cam, pipe, G, aux=None):
    from gaussian_renderer import render
    pkg = render(cam, model, pipe, torch.zeros(3, device=DEV))
    loss = (pkg["render"] * G).sum()
    if aux is not None:
        loss = loss + (pkg["depth"] * aux[0]).sum() + (pkg["alpha"] * aux[1]).sum()
    loss.backward()
    return pkg


@pytest.mark.parametrize("name,aux", [("small", False), ("rotcam", True), ("dur10", False), ("smod2", False), ("dim3", False),
                                      ("norot4d", False), ("deg1m4", False), ("mid", False)])
def test_fused_prologue_matches_getter_path(name, aux):
    cfg, cam, sc, st = helpers.build(name, device=DEV)
    cam = cam.to(DEV)
    gc, gd, ga, gf = helpers.pixel_grads(cfg, device=DEV)
    A = RawModel(sc, seed=1, requires_grad=True)
    B = RawModel(sc, seed=1, requires_grad=True)
    # scale_modifier / prefilter are per-call settings of render(); the configuration's modifier is applied to both
    pa = _render_and_backward(A, cam, PipeUnfused(), gc, (gd, ga) if aux else None)
    pb = _render_and_backward(B, cam, Pipe(), gc, (gd, ga) if aux else None)
    same_radii = (pa["radii"] == pb["radii"]).float().mean().item()
    assert same_radii > 0.9995, same_radii
    assert helpers.psnr(helpers.to_np(pb["render"]), helpers.to_np(pa["render"])) > 90.0
    assert helpers.max_rel(helpers.to_np(pb["depth"]), helpers.to_np(pa["depth"])) < 1e-4
    print("%s: image bit-identical: %s, radii identical: %.6f" % (name, torch.equal(pa["render"], pb["render"]), same_radii))
    for k, a in A.leaves().items():
        b = B.leaves()[k]
        if a.grad is None:
            assert b.grad is None or float(b.grad.abs().max()) == 0.0, k
            continue
        assert b.grad is not None and b.grad.shape == a.grad.shape, k
        err = helpers.l2_rel(helpers.to_np(b.grad), helpers.to_np(a.grad))
        # both sides run the same (non-deterministic) blend backward: blend-level tensors agree to its noise; the
        # covariance chain amplifies that noise (see test_gpu_parity.py) -- at 100k Gaussians up to a few 1e-4
        assert err < (2e-3 if (k in CHAIN and cfg["P"] >= 50000) else 1e-4), (k, err)
    assert helpers.l2_rel(helpers.to_np(pb["viewspace_points"].grad), helpers.to_np(pa["viewspace_points"].grad)) < 1e-4


def test_raw_entry_vs_reference_render_at_cfg3():
    """VERDICT r1 next #4: gradients w.r.t. the RAW parameters against the reference rasterizer under the reference's
    own torch prologue (getters + autograd), at cfg3.  Blend-level / SH / position tensors to 1e-4; the covariance chain
    against the reference's own run-to-run spread (it is not reproducible to 1e-4 at this size).  The reference's three
    runs are a record (tests/golden/ref_raw_cfg3.npz, tools/ref_golden.py): a pixel sample of its image, and per leaf
    the mean gradient on a sample of rows with the runs' spread there and over the whole tensor."""
    rec = helpers.ref_record("raw_cfg3")
    cfg, cam, sc, st = helpers.build("cfg3", device=DEV)
    cam = cam.to(DEV)
    g = torch.Generator().manual_seed(77)
    G = torch.randn(3, cfg["H"], cfg["W"], generator=g).to(DEV)
    B = RawModel(sc, seed=2, requires_grad=True)
    pb = _render_and_backward(B, cam, Pipe(), G)
    pix = torch.from_numpy(rec["pixels"]).long().to(DEV)
    assert helpers.psnr(helpers.to_np(pb["render"].reshape(3, -1)[:, pix]), rec["image"]) > 90.0
    for k, b in B.leaves().items():
        s, m, norm_dev, st = helpers.grad_sample(rec[k], b.grad)
        l2 = ((s - m).norm() / m.norm()).item()
        # the runs' spread over the whole tensor or on the sample, whichever is larger: on the covariance chain a few
        # noisy rows outside the sample carry most of the whole tensor's spread
        spread = max(st["l2max"], st["l2max_full"])
        assert l2 < max(1e-4, 4 * spread), (k, l2, spread)
        assert norm_dev < max(1e-4, 4 * st["l2max_full"]), (k, "norm", norm_dev, st["l2max_full"])
        print("raw grad %-13s vs reference render(): l2 %.2e (reference spread %.2e)" % (k, l2, spread))


def test_view_parallel_step_with_raw_entry():
    """factor mode + raw entry on one GPU: 3 views, gradients at the raw leaves == sequential autograd accumulation"""
    from fdgs.dist import ViewParallelStep
    from gaussian_renderer import render
    import test_gpu_view_parallel as vp
    cfg, cam, sc, st = helpers.build("n3v", device=DEV)
    cams = vp._views(cfg, 3, DEV)
    bg = torch.zeros(3, device=DEV)
    A = RawModel(sc, seed=4, requires_grad=True)
    B = RawModel(sc, seed=4, requires_grad=True)
    Gs = [torch.randn(3, cfg["H"], cfg["W"], generator=torch.Generator().manual_seed(50 + k)).to(DEV) for k in range(3)]
    for k, c in enumerate(cams):
        ((render(c, A, Pipe(), bg)["render"] * Gs[k]).sum() / 3).backward()
    step = ViewParallelStep(sc.P, DEV)
    with step:
        for k, c in enumerate(cams):
            pkg = render(c, B, Pipe(), bg)
            ((pkg["render"] * Gs[k]).sum() / 3).backward()
            step.add_view_stats(pkg["viewspace_points"].grad, pkg["radii"])
    lv = B.leaves()
    step.finish([lv[k] for k in ("xyz", "t", "scaling", "scaling_t", "rotation", "rotation_r", "opacity")],
                [lv["features_dc"], lv["features_rest"]])
    for k, a in A.leaves().items():
        assert helpers.l2_rel(helpers.to_np(lv[k].grad), helpers.to_np(a.grad)) < (2e-6 if k.startswith("features") else 1e-4), k
