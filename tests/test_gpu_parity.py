"""GPU (-m gpu): the parity tests proper.  Everything goes through the reference-facing boundary
(the `_C`-compatible extension over the C-ABI, and the GaussianRasterizer / render() API on top).

Three checkers, strongest first:
  1. golden vectors produced by the UNMODIFIED reference kernels (tests/golden/*.npz)  -> bit-exact
     forward (every tensor), gradients within the reference's own atomic-order noise;
  2. records of the compiled reference at the BASELINE sizes (500k / 2M Gaussians, 1352x1014;
     tests/golden/ref_*.npz, written by tools/ref_golden.py)                            -> same bar;
  3. the CPU oracle on seeded inputs the oracle finishes in seconds, including the branches the
     golden set does not cover (3D Gaussians, 3D SH, no-rot 4D, low SH degree, M=16, prefilter,
     ragged image sizes, precomputed colours / covariances).
Plus size-independent properties at full size: sortedness of the instance list, range
consistency, run-to-run determinism of the forward, linearity and locality of the backward.
"""
import numpy as np
import pytest
import torch

import helpers
import oracle_py

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


@pytest.fixture(scope="module")
def C():
    import fdgs
    return fdgs.ext()   # raises if the CUDA extension is missing -- there is no fallback path


# Gradient bar (north_star: 1e-4 relative fp32).  The reference accumulates with unordered fp32 atomics, so a
# single reference run is a noisy sample; so is ours (RED order, reassociated sums).  Our gradients are compared with
# the MEAN of K reference reruns; if ours is "one more sample of the same quantity" its distance to that mean is
# about one per-run spread (sqrt(1 + 1/K) of it).  Bar per tensor, in the L2 and in the max-norm sense:
#     err(ours, mean) < max(1e-4, 4 * spread)             (max-norm: 5 * spread)
# i.e. 1e-4 wherever the reference itself is reproducible to 1e-4 (all blend-level, SH and mean gradients, at every
# size), and "statistically indistinguishable from a reference rerun" for the covariance chain (division by cov_t^2
# and near-singular determinants amplify the 1e-7 upstream noise ~1000x: the reference's own spread reaches 3e-3 on
# dL_dscales_t at 2M Gaussians, and the deterministic serial-sum oracle and the reference mean differ by 3e-4 on
# dL_drot at 100k -- profiles/r02_parity_table.md).  That table is the evidence; no fp32 implementation pins those
# four tensors to 1e-4 at scale.
# The reference's 8 reruns are stored as a record (tests/helpers.py: grad_record): their mean on a seeded sample of rows
# (the largest rows and random ones), the spreads on that sample, and the norm and spread of the whole tensor.  The
# bars apply on the sample; the norm of our whole tensor must match the reference mean's within the L2 bar.


def check_grad_vs_reference(gname, a, rec):
    if rec[gname].size == 1 and rec[gname][0] == helpers.GRAD_ZERO:
        assert float(a.abs().max()) == 0.0, gname
        return
    s, m, norm_dev, st = helpers.grad_sample(rec[gname], a)
    # the reference's spread over the whole tensor or on the sample, whichever is larger: a few noisy rows outside the
    # sample can carry most of the whole tensor's spread (covariance chain)
    l2n, mxn = max(st["l2n"], st["l2n_full"]), st["mxn"]
    nm, sc = m.norm().item(), m.abs().max().item()
    l2 = ((s - m).norm() / nm).item()
    err = (s - m).abs().max().item() / sc
    chain = gname in ("dL_dts", "dL_dscales", "dL_dscales_t", "dL_drot", "dL_drot_r", "dL_dcov3D")
    if st["l2n_full"] < 2e-4 and not (chain and st["l2n_full"] > 1e-5):
        assert norm_dev < max(1e-4, 4 * st["l2n_full"]), (gname, "norm", norm_dev, "ref spread", st["l2n_full"])
        assert l2 < max(1e-4, 4 * l2n), (gname, "l2", l2, "ref spread", l2n)
        assert err < max(1e-4, 5 * mxn), (gname, "max", err, "ref spread", mxn)
    else:
        # (Covariance-chain tensors whose reference spread is already above 1e-5 take this branch too: their norm
        # error is a heavy-tailed statistic -- for ONE configuration and code version, three of our runs and three
        # estimates of the reference's spread from 8 reruns each scattered over 4.3e-5 ... 7.3e-5 and 4.1e-5 ... 5.4e-5
        # on dL_dts, profiles/r02_grad_noise_probe.txt -- so the norm gets 6 spreads and the rows carry the check.)
        # The reference does not reproduce ITSELF to 0.02 % here (cfg5's long time axis: a handful of Gaussians with
        # near-singular conditional covariances carry most of the norm and amplify the atomics' rounding noise to
        # 5-30 %, profiles/r02_parity_table.md).  Norms are then heavy-tailed statistics of a few rows: keep a loose
        # norm bound and check the well-conditioned majority row by row instead.
        assert norm_dev < max(1e-4, 6 * st["l2n_full"]), (gname, "norm", norm_dev, "ref spread", st["l2n_full"])
        assert l2 < max(1e-4, 6 * l2n), (gname, "l2", l2, "ref spread", l2n)
        ours_med = helpers.median_row_err(s, m)
        ref_med = st["rmed"]
        assert ours_med < max(1e-4, 3 * ref_med), (gname, "median row error", ours_med, "reference runs", ref_med)


@pytest.fixture(params=[1, 0], ids=["tilecull", "reflists"])
def tile_mode(request):
    """1 = the library's default tile lists (only instances a pixel can blend), 0 = the reference's lists exactly
    (include/fdgs.h: fdgs_set_tile_cull)."""
    import fdgs
    prev = fdgs.set_tile_cull(request.param)
    yield request.param
    fdgs.set_tile_cull(prev)


def lists_of(o):
    return dict(point_list=helpers.to_np(o["point_list"]), ranges=helpers.to_np(o["ranges"]),
                n_contrib=helpers.to_np(o["n_contrib"]).reshape(-1), num_rendered=int(o["fw"][0]))


def run_cuda(C, name_or_cfg, with_backward=True, grads=None):
    cfg, cam, sc, st = helpers.build(name_or_cfg, device=DEV)
    fw = C.rasterize_gaussians(*helpers.fwd_args(st, sc, cfg))
    out = dict(cfg=cfg, sc=sc, st=st, fw=fw)
    P, W, H = cfg["P"], cfg["W"], cfg["H"]
    geom = C.debug_export_geom(fw[6], P)
    binning = C.debug_export_binning(fw[7], fw[8], fw[0], W, H)
    out.update(depths=geom[0], means2D=geom[1], conic_opacity=geom[2], rgb=geom[3], clamped=geom[4], tiles=geom[5],
               point_list=binning[0], ranges=binning[1], n_contrib=binning[2])
    if with_backward:
        grads = grads if grads is not None else helpers.pixel_grads(cfg, device=DEV)
        out["grads_in"] = grads
        out["bw"] = C.rasterize_gaussians_backward(*helpers.bwd_args(st, sc, cfg, fw, grads))
    torch.cuda.synchronize()
    return out


def clamp_bits_to_bools(c):
    return torch.stack([(c >> i) & 1 for i in range(3)], 1)


# ---------------------------------------------------------------------------------------------------
# 1. golden vectors from the reference kernels
# ---------------------------------------------------------------------------------------------------
GOLDEN_CASES = ["tiny", "small", "flowbg", "negfov", "ragged", "sh3d", "dim3", "norot4d", "deg1", "m16", "prefilter",
                "dur10", "smod05", "smod2", "rotcam", "n3v", "deg1m4"]


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_forward_bit_exact_vs_golden(C, name, tile_mode):
    G = helpers.golden(name)
    if G is None:
        pytest.skip("no golden fixture for %s" % name)
    o = run_cuda(C, name, with_backward=False)
    fw = o["fw"]
    np_ = helpers.to_np
    assert helpers.bitdiff(np_(fw[5]), G["radii"]) == 0
    helpers.check_tile_lists(lists_of(o), dict(point_list=G["point_list"], ranges=G["ranges"], n_contrib=G["n_contrib"],
                                               num_rendered=int(G["num_rendered"])), o["cfg"]["W"], o["cfg"]["H"], tile_mode)
    vis = G["radii"] > 0
    assert helpers.bitdiff(np_(o["tiles"]), G["tiles_touched"]) == 0
    assert helpers.bitdiff(np_(fw[10]), G["out_means3D"]) == 0
    for ours, ref in ((o["depths"], "depths"), (o["means2D"], "means2D"), (o["conic_opacity"], "conic_opacity"),
                      (o["rgb"], "rgb"), (fw[9], "covs3D")):
        assert helpers.bitdiff(np_(ours)[vis], G[ref][vis]) == 0, ref
    assert helpers.bitdiff(np_(clamp_bits_to_bools(o["clamped"]))[vis], G["clamped"][vis]) == 0
    for idx, key in ((1, "color"), (2, "flow"), (3, "depth"), (4, "T")):
        assert helpers.bitdiff(np_(fw[idx]), G[key]) == 0, key


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_backward_vs_golden(C, name):
    G = helpers.golden(name)
    if G is None:
        pytest.skip("no golden fixture for %s" % name)
    o = run_cuda(C, name)
    for gname, ours in zip(helpers.GRAD_NAMES, o["bw"]):
        ref = G["grad_" + gname]
        if ref.size == 0:
            continue
        a = helpers.to_np(ours).reshape(ref.shape)
        # the reference accumulates with unordered fp32 atomics: norm-wise 1e-4, max-norm looser
        assert helpers.l2_rel(a, ref) < 1e-4, gname
        assert helpers.max_rel(a, ref) < 2e-3, gname


@pytest.mark.parametrize("name", ["small", "flowbg", "sh3d", "mid"])
def test_colour_only_backward_equals_zero_aux_gradients(C, name):
    """No upstream gradient for depth / alpha / flow (NULL in the C-ABI, None in autograd) selects the
    9-value blend-backward instantiation; it must agree with the general one fed explicit zeros."""
    cfg, cam, sc, st = helpers.build(name, device=DEV)
    gc, gd, ga, gf = helpers.pixel_grads(cfg, device=DEV)
    fw = C.rasterize_gaussians(*helpers.fwd_args(st, sc, cfg))
    e = torch.empty(0, device=DEV)
    lean = C.rasterize_gaussians_backward(*helpers.bwd_args(st, sc, cfg, fw, (gc, e, e, e)))
    full = C.rasterize_gaussians_backward(*helpers.bwd_args(st, sc, cfg, fw, (gc, 0 * gd, 0 * ga, 0 * gf)))
    again = C.rasterize_gaussians_backward(*helpers.bwd_args(st, sc, cfg, fw, (gc, 0 * gd, 0 * ga, 0 * gf)))
    for gname, a, b, b2 in zip(helpers.GRAD_NAMES, lean, full, again):
        if b.numel() == 0:
            continue
        assert torch.isfinite(a).all(), gname
        # tolerance: the run-to-run noise of the unordered fp32 atomics (amplified by the covariance
        # chain for scales / rotations) or 2e-5, whichever is larger
        noise = helpers.l2_rel(helpers.to_np(b2), helpers.to_np(b))
        assert helpers.l2_rel(helpers.to_np(a), helpers.to_np(b)) < max(2e-5, 8 * noise), (gname, noise)
    assert float(lean[helpers.GRAD_NAMES.index("dL_dflows")].abs().max()) == 0.0
    # a single missing image is handled by the general instantiation
    part = C.rasterize_gaussians_backward(*helpers.bwd_args(st, sc, cfg, fw, (gc, gd, e, gf)))
    ref = C.rasterize_gaussians_backward(*helpers.bwd_args(st, sc, cfg, fw, (gc, gd, 0 * ga, gf)))
    ref2 = C.rasterize_gaussians_backward(*helpers.bwd_args(st, sc, cfg, fw, (gc, gd, 0 * ga, gf)))
    for gname, a, b, b2 in zip(helpers.GRAD_NAMES, part, ref, ref2):
        if b.numel():
            noise = helpers.l2_rel(helpers.to_np(b2), helpers.to_np(b))
            assert helpers.l2_rel(helpers.to_np(a), helpers.to_np(b)) < max(2e-5, 8 * noise), (gname, noise)


@pytest.mark.parametrize("P,expect_min", [(4000, 0), (30000, 2049), (200000, 16385)])
def test_tile_lists_sorted_and_complete(C, P, expect_min, tile_mode):
    """Every path of the per-tile sort (<= 2048 keys: 8 keys per thread; <= 16384: the large
    shared-memory instantiation; above: in place in global memory) must produce, for every tile,
    exactly the instances whose tile rectangle covers it, ordered by (depth bits, Gaussian index) --
    the order the reference's stable radix sort of tile|depth keys gives (rasterizer_impl.cu:325)."""
    cfg = dict(P=P, W=32, H=32, seed=4242 + P)
    o = run_cuda(C, cfg, with_backward=False)
    radii = helpers.to_np(o["fw"][5]).astype(np.int64)
    px = helpers.to_np(o["means2D"])[:, 0].astype(np.float32)
    py = helpers.to_np(o["means2D"])[:, 1].astype(np.float32)
    depth_bits = helpers.to_np(o["depths"]).astype(np.float32).view(np.uint32).astype(np.uint64)
    ranges = helpers.to_np(o["ranges"]).reshape(-1, 2).astype(np.int64)
    plist = helpers.to_np(o["point_list"]).astype(np.int64)
    con = helpers.to_np(o["conic_opacity"])
    gx = gy = 2
    r = radii.astype(np.float32)
    f = np.float32
    x0 = np.clip(((px - r) * f(0.0625)).astype(np.int64), 0, gx)
    y0 = np.clip(((py - r) * f(0.0625)).astype(np.int64), 0, gy)
    x1 = np.clip(((((px + r) + f(16.0)) + f(-1.0)) * f(0.0625)).astype(np.int64), 0, gx)
    y1 = np.clip(((((py + r) + f(16.0)) + f(-1.0)) * f(0.0625)).astype(np.int64), 0, gy)
    vis = radii > 0
    if tile_mode == 0:
        assert (ranges[:, 1] - ranges[:, 0]).max() >= expect_min, "configuration does not reach the intended sort path"
    assert (ranges[:, 1] - ranges[:, 0]).sum() == int(o["fw"][0]) == len(plist)
    for ty in range(gy):
        for tx in range(gx):
            lo, hi = ranges[ty * gx + tx]
            ids = plist[lo:hi]
            want = np.nonzero(vis & (x0 <= tx) & (tx < x1) & (y0 <= ty) & (ty < y1))[0]
            key = (depth_bits[want] << np.uint64(32)) | want.astype(np.uint64)
            want = want[np.argsort(key, kind="stable")]
            if tile_mode == 0:
                assert len(ids) == len(want)
                assert (ids == want).all()
                continue
            # default lists: the reference's list with instances removed, order kept ...
            keep = np.isin(want, ids)
            assert int(keep.sum()) == len(ids) and (want[keep] == ids).all()
            # ... and no pixel of the tile reaches alpha = 1/255 for a removed instance (float64, 1 % margin; the cull
            # keeps 2 % of slack)
            gone = want[~keep]
            xs = (np.arange(16) + 16 * tx).astype(np.float64)
            ys = (np.arange(16) + 16 * ty).astype(np.float64)
            for lo_g in range(0, len(gone), 20000):
                gsel = gone[lo_g:lo_g + 20000]
                cx, cy = px[gsel].astype(np.float64), py[gsel].astype(np.float64)
                A, B, Cc, op_ = (con[gsel, i].astype(np.float64) for i in range(4))
                dx = cx[:, None, None] - xs[None, None, :]
                dy = cy[:, None, None] - ys[None, :, None]
                power = -0.5 * (A[:, None, None] * dx * dx + Cc[:, None, None] * dy * dy) - B[:, None, None] * dx * dy
                alpha = op_[:, None, None] * np.exp(np.minimum(power, 0.0))
                assert not ((power <= 0) & (alpha >= (1.0 / 255.0) * 0.99)).any(), "a removed instance had a contributing pixel"
    if tile_mode == 1 and P >= 30000:
        assert int(o["fw"][0]) < (x1 - x0)[vis].dot((y1 - y0)[vis]), "tile culling removed nothing"


# ---------------------------------------------------------------------------------------------------
# 2. the compiled reference at BASELINE sizes
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["mid", "mid_rotcam", "mid_dur10", "mid_smod2", "cfg5", "cfg2", "cfg3"])
def test_full_size_vs_compiled_reference(C, name, tile_mode):
    rec = helpers.ref_record("full_" + name)
    o = run_cuda(C, name)
    cfg, sc, st, fw = o["cfg"], o["sc"], o["st"], o["fw"]
    P, W, H = cfg["P"], cfg["W"], cfg["H"]
    assert helpers.digest(fw[5]) == rec["radii"]                             # radii
    # tile assignment + order, last contributors: the reference-list mode reproduces the reference's lists bit for
    # bit, and the default lists are checked against those
    ours = lists_of(o)
    if tile_mode == 0:
        ref_lists = ours
    else:
        import fdgs
        with fdgs.tile_cull(0):
            fw0 = C.rasterize_gaussians(*helpers.fwd_args(st, sc, cfg))
            b0 = C.debug_export_binning(fw0[7], fw0[8], fw0[0], W, H)
        ref_lists = dict(point_list=helpers.to_np(b0[0]), ranges=helpers.to_np(b0[1]),
                         n_contrib=helpers.to_np(b0[2]).reshape(-1), num_rendered=int(fw0[0]))
        del fw0, b0
    for k, v in helpers.list_digests(ref_lists).items():
        assert v == rec[k], k
    helpers.check_tile_lists(ours, ref_lists, W, H, tile_mode)
    for i, key in ((1, "color"), (2, "flow"), (3, "depth"), (4, "T"), (10, "out_means3D")):
        assert helpers.digest(fw[i]) == rec[key], key
    assert helpers.digest(fw[9][fw[5] > 0]) == rec["cov3D"]
    for gname, a in zip(helpers.GRAD_NAMES, o["bw"]):
        if rec[gname][0] == helpers.GRAD_EMPTY:
            continue
        check_grad_vs_reference(gname, a, rec)


@pytest.mark.parametrize("name", ["small", "ragged", "negfov", "rotcam", "n3v", "mid", "mid_dur10", "cfg5", "cfg2", "cfg3"])
def test_colour_only_backward_vs_compiled_reference(C, name):
    """The training default: only the colour image carries a gradient.  That selects the tensor-core
    blend-backward (polynomial power + mma reduction, blend_bwd.cu v2); the reference gets explicit
    zero images for depth / alpha / flow.  Same bar as the general path: 1e-4 in the L2 sense or a few
    times the reference's own run-to-run atomic noise."""
    rec = helpers.ref_record("colour_" + name)
    cfg, cam, sc, st = helpers.build(name, device=DEV)
    gc, gd, ga, gf = helpers.pixel_grads(cfg, device=DEV)
    e = torch.empty(0, device=DEV)
    fw = C.rasterize_gaussians(*helpers.fwd_args(st, sc, cfg))
    ours = C.rasterize_gaussians_backward(*helpers.bwd_args(st, sc, cfg, fw, (gc, e, e, e)))
    torch.cuda.synchronize()
    for gname, a in zip(helpers.GRAD_NAMES, ours):
        if rec[gname][0] == helpers.GRAD_EMPTY:
            continue
        assert torch.isfinite(a).all(), gname
        check_grad_vs_reference(gname, a, rec)


# ---------------------------------------------------------------------------------------------------
# 3. the CPU oracle, including branches without golden coverage
# ---------------------------------------------------------------------------------------------------
ORACLE_CASES = ["tiny", "flowbg", "negfov", "ragged", "sh3d", "dim3", "norot4d", "deg1", "m16", "prefilter",
                "dur10", "smod05", "smod2", "rotcam", "n3v", "deg1m4",
                "mid", "mid_rotcam", "q250k"]       # deterministic (serial-sum) 1e-4 pin of all 12 gradients at scale


@pytest.mark.parametrize("name", ORACLE_CASES)
def test_vs_cpu_oracle(C, name, tile_mode):
    o = run_cuda(C, name)
    cfg, fw = o["cfg"], o["fw"]
    cfg_c, cam, sc_c, st_c = helpers.build(name)
    inp = helpers.oracle_inputs(st_c, sc_c, cfg_c)
    f = oracle_py.forward(inp)
    np_ = helpers.to_np
    assert helpers.bitdiff(np_(fw[5]), f["radii"]) == 0
    if tile_mode == 0:
        assert fw[0] == f["num_rendered"]
        assert helpers.bitdiff(np_(o["point_list"]), f["point_list"]) == 0
        assert helpers.bitdiff(np_(o["ranges"]), f["ranges"]) == 0
    else:
        assert fw[0] <= f["num_rendered"]      # the shorter lists are compared with the reference's in the tests above
    vis = f["radii"] > 0
    assert helpers.bitdiff(np_(fw[10]), f["out_means3D"]) == 0
    for ours, key in ((o["depths"], "depths"), (o["means2D"], "means2D"), (o["rgb"], "rgb"), (fw[9], "cov3D")):
        assert helpers.bitdiff(np_(ours)[vis], f[key][vis]) == 0, key
    assert helpers.bitdiff(np_(o["conic_opacity"])[vis][:, :3], f["conic_opacity"][vis][:, :3]) == 0
    assert helpers.max_rel(np_(o["conic_opacity"])[vis][:, 3], f["conic_opacity"][vis][:, 3]) < 1e-6   # MUFU vs libm
    # n_contrib can only differ where CUDA's expf and libm's land on opposite sides of a blend threshold
    if tile_mode == 0:
        assert helpers.bitdiff(np_(o["n_contrib"]), f["n_contrib"]) <= max(2, cfg["W"] * cfg["H"] // 20000)
    for idx, key in ((1, "color"), (2, "flow"), (3, "depth")):
        assert helpers.max_rel(np_(fw[idx]), f[key]) < 1e-5, key
    assert helpers.psnr(np_(fw[1]), f["color"]) > 100
    g = oracle_py.backward(inp, f, *[np_(t) for t in o["grads_in"]])
    for gname, okey, ours in zip(helpers.GRAD_NAMES, helpers.ORACLE_GRAD_KEYS, o["bw"]):
        ref = g[okey]
        if ref.size == 0:
            continue
        a = np_(ours).reshape(ref.shape)
        # 1e-4 everywhere, except the covariance-chain tensors at scale: there the serial-sum oracle and the mean of
        # reference runs themselves differ by ~3e-4 (profiles/r02_parity_table.md, column "ref-mean vs oracle")
        # (the long-time-axis cases dur10 / n3v sit at 1.1e-4 on dL_dscales_t already at 3000 Gaussians)
        chain = gname in ("dL_dts", "dL_dscales", "dL_dscales_t", "dL_drot", "dL_drot_r", "dL_dcov3D")
        big = cfg["P"] >= 50000
        assert helpers.l2_rel(a, ref) < ((1e-3 if big else 3e-4) if chain else 1e-4), gname
        assert helpers.max_rel(a, ref) < (2e-2 if (chain and big) else 1e-3), gname


def test_precomputed_colors_and_covariance_vs_oracle(C):
    """colors_precomp / cov3D_precomp branches (reference: forward.cu:411-414,476; backward.cu:897,908)."""
    cfg, cam, sc, st = helpers.build("tiny", device=DEV)
    cfg_c, _, sc_c, st_c = helpers.build("tiny")
    g = torch.Generator().manual_seed(3)
    colors = torch.rand(cfg["P"], 3, generator=g)
    A = 0.05 * torch.randn(cfg["P"], 3, 3, generator=g)
    cov = A @ A.transpose(1, 2) + 1e-4 * torch.eye(3)
    cov6 = torch.stack([cov[:, 0, 0], cov[:, 0, 1], cov[:, 0, 2], cov[:, 1, 1], cov[:, 1, 2], cov[:, 2, 2]], 1).contiguous()
    e = torch.Tensor([])
    args = (st["bg"], sc.means3D, colors.to(DEV), sc.flow_2d, sc.opacities, e, e, e, e, e, 1.0, cov6.to(DEV), -1.0,
            st["viewmatrix"], st["projmatrix"], st["tanfovx"], st["tanfovy"], cfg["H"], cfg["W"], e, 0, 0, st["campos"],
            st["timestamp"], st["time_duration"], False, 3, False, False, False)
    fw = C.rasterize_gaussians(*args)
    st3 = dict(st_c)
    st3.update(rot_4d=False, gaussian_dim=3, sh_degree=0, sh_degree_t=0)
    inp = oracle_py.OracleInputs(st3, sc_c.means3D, sc_c.opacities, colors_precomp=colors, flow_2d=sc_c.flow_2d,
                                 cov3D_precomp=cov6)
    f = oracle_py.forward(inp)
    np_ = helpers.to_np
    import fdgs
    with fdgs.tile_cull(0):
        assert C.rasterize_gaussians(*args)[0] == f["num_rendered"]     # the reference's tile lists
    assert fw[0] <= f["num_rendered"]                                   # default lists: only instances a pixel can blend
    assert helpers.bitdiff(np_(fw[5]), f["radii"]) == 0
    assert helpers.max_rel(np_(fw[1]), f["color"]) < 1e-5
    grads = helpers.pixel_grads(cfg, device=DEV)
    (num_rendered, color, flow, depth, T, radii, geom, binning, img, covs, out_means3D) = fw
    bw = C.rasterize_gaussians_backward(st["bg"], sc.means3D, out_means3D, radii, colors.to(DEV), sc.flow_2d, sc.opacities,
                                        e, e, e, e, e, 1.0, cov6.to(DEV), -1.0, st["viewmatrix"], st["projmatrix"],
                                        st["tanfovx"], st["tanfovy"], *grads, e, 0, 0, st["campos"], st["timestamp"],
                                        st["time_duration"], False, 3, False, geom, num_rendered, binning, img, False)
    go = oracle_py.backward(inp, f, *[np_(t) for t in grads])
    for gname, okey, ours in zip(helpers.GRAD_NAMES, helpers.ORACLE_GRAD_KEYS, bw):
        ref = go[okey]
        if ref.size == 0 or gname in ("dL_dsh",):
            continue
        assert helpers.l2_rel(np_(ours).reshape(ref.shape), ref) < 1e-4, gname


def test_empty_and_degenerate_inputs(C):
    cfg, cam, sc, st = helpers.build("tiny", device=DEV)
    # P = 0 (reference: rasterize_points.cu:97,215)
    sc0 = helpers.synth.make_scene(0, cam, 1).to(DEV)
    fw = C.rasterize_gaussians(*helpers.fwd_args(st, sc0, cfg))
    assert fw[0] == 0 and fw[5].numel() == 0
    assert torch.all(fw[4] == 1.0) and torch.all(fw[1] == 0.0)
    # everything behind the camera / outside the time window: nothing rendered, background only
    sc1 = helpers.build("tiny", device=DEV)[2]
    sc1.means3D[:, 2] = -5.0
    st_bg = dict(st)
    st_bg["bg"] = torch.tensor([0.1, 0.2, 0.3], device=DEV)
    fw = C.rasterize_gaussians(*helpers.fwd_args(st_bg, sc1, cfg))
    assert fw[0] == 0 and int((fw[5] > 0).sum()) == 0
    assert torch.allclose(fw[1][:, 5, 7], torch.tensor([0.1, 0.2, 0.3], device=DEV))
    grads = helpers.pixel_grads(cfg, device=DEV)
    bw = C.rasterize_gaussians_backward(*helpers.bwd_args(st_bg, sc1, cfg, fw, grads))
    assert all(float(t.abs().sum()) == 0.0 for t in bw)
    # mark_visible (reference: rasterizer_impl.cu:54-67)
    vis = C.mark_visible(sc.means3D, st["viewmatrix"], st["projmatrix"])
    assert torch.equal(vis, sc.means3D[:, 2] > 0.2)


# ---------------------------------------------------------------------------------------------------
# size-independent properties at the BASELINE size
# ---------------------------------------------------------------------------------------------------
def test_full_size_properties(C):
    o = run_cuda(C, "cfg3")
    cfg, fw = o["cfg"], o["fw"]
    R = fw[0]
    P, W, H = cfg["P"], cfg["W"], cfg["H"]
    # the lists hold only instances a pixel can blend (fdgs_set_tile_cull, default): never more than the reference's
    # tile rectangles (tiles_touched keeps the reference's count), and far fewer on this scene
    assert R <= int(o["tiles"].long().sum())
    import fdgs
    with fdgs.tile_cull(0):
        fw_ref_lists = C.rasterize_gaussians(*helpers.fwd_args(o["st"], o["sc"], cfg))
    assert fw_ref_lists[0] == int(o["tiles"].long().sum())
    for i in (1, 2, 3, 4, 5, 10):     # colour, flow, depth, T, radii, out_means3D: independent of the list mode
        assert torch.equal(fw[i], fw_ref_lists[i]), i
    del fw_ref_lists
    ranges = o["ranges"].long()
    pl = o["point_list"].long()
    # ranges tile the instance list exactly
    nonempty = ranges[:, 1] > ranges[:, 0]
    starts = ranges[nonempty, 0]
    ends = ranges[nonempty, 1]
    assert int(starts[0]) == 0 and int(ends[-1]) == R and torch.equal(starts[1:], ends[:-1])
    # within every tile the list is sorted by (depth bits, Gaussian index): a checksum-free sortedness test
    depth_bits = o["depths"].view(torch.int32).long()[pl]
    tile_of = torch.repeat_interleave(torch.arange(ranges.shape[0], device=DEV), (ranges[:, 1] - ranges[:, 0]))
    key = (tile_of << 32) | depth_bits
    assert bool(torch.all(key[1:] >= key[:-1]))
    same = key[1:] == key[:-1]
    assert bool(torch.all(pl[1:][same] > pl[:-1][same]))
    # n_contrib never exceeds the tile's list length
    gx = (W + 15) // 16
    ys, xs = torch.meshgrid(torch.arange(H, device=DEV), torch.arange(W, device=DEV), indexing="ij")
    tl = (ys // 16) * gx + xs // 16
    assert bool(torch.all(o["n_contrib"].long() <= (ranges[:, 1] - ranges[:, 0])[tl]))
    # forward is deterministic: bit-identical on a second run
    o2 = run_cuda(C, "cfg3", with_backward=False)
    for i in (1, 2, 3, 4, 5, 10):
        assert torch.equal(fw[i], o2["fw"][i])
    # backward: linear in the upstream gradients, zero in -> zero out, nothing for unrendered Gaussians
    g1 = o["grads_in"]
    g2 = tuple(torch.randn_like(t) for t in g1)
    st, sc = o["st"], o["sc"]
    b2 = C.rasterize_gaussians_backward(*helpers.bwd_args(st, sc, cfg, fw, g2))
    b12 = C.rasterize_gaussians_backward(*helpers.bwd_args(st, sc, cfg, fw, tuple(2.0 * a - 0.5 * b for a, b in zip(g1, g2))))
    bz = C.rasterize_gaussians_backward(*helpers.bwd_args(st, sc, cfg, fw, tuple(torch.zeros_like(t) for t in g1)))
    invisible = fw[5] <= 0
    for name, a, b, ab, z in zip(helpers.GRAD_NAMES, o["bw"], b2, b12, bz):
        lin = 2.0 * a - 0.5 * b
        # linear up to fp32 round-off; the ill-conditioned covariance chain amplifies it (the reference's
        # own run-to-run noise on dL_dscales_t / dL_drot is ~1e-2 in max-norm at this size)
        assert ((ab - lin).double().norm() / lin.double().norm()).item() < 3e-2, name
        assert float(z.abs().sum()) == 0.0, name
        assert float(a[invisible].abs().sum()) == 0.0, name


# ---------------------------------------------------------------------------------------------------
# the Python API on top (GaussianRasterizer + render()), autograd end to end
# ---------------------------------------------------------------------------------------------------
class _Model:
    """Duck-typed stand-in for the reference's GaussianModel getters (scene/gaussian_model.py:179-251)."""

    def __init__(self, sc):
        self.sc = sc
        self.get_xyz = sc.means3D.clone().requires_grad_(True)
        self.get_opacity = sc.opacities.clone().requires_grad_(True)
        self.get_scaling = sc.scales.clone().requires_grad_(True)
        self.get_scaling_t = sc.scales_t.clone().requires_grad_(True)
        self.get_rotation = sc.rotations.clone().requires_grad_(True)
        self.get_rotation_r = sc.rotations_r.clone().requires_grad_(True)
        self.get_t = sc.ts.clone().requires_grad_(True)
        self.get_features = sc.shs.clone().requires_grad_(True)
        self.active_sh_degree, self.active_sh_degree_t = sc.sh_degree, sc.sh_degree_t
        self.time_duration = [0.0, sc.time_duration]
        self.rot_4d, self.gaussian_dim, self.force_sh_3d = sc.rot_4d, sc.gaussian_dim, sc.force_sh_3d
        self.prefilter_var = -1.0
        self.get_max_sh_channels = sc.shs.shape[1]


class _Pipe:
    convert_SHs_python = False
    compute_cov3D_python = False
    debug = False
    env_map_res = 0


def test_render_api_end_to_end(C):
    from gaussian_renderer import render
    cfg, cam, sc, st = helpers.build("small", device=DEV)
    pc = _Model(sc)
    bg = torch.zeros(3, device=DEV)
    pkg = render(cam.to(DEV), pc, _Pipe(), bg)
    assert set(pkg) == {"render", "viewspace_points", "visibility_filter", "radii", "depth", "alpha", "flow"}
    G = helpers.golden("small")
    assert helpers.bitdiff(helpers.to_np(pkg["render"]), G["color"]) == 0
    assert helpers.bitdiff(helpers.to_np(pkg["radii"]), G["radii"]) == 0
    assert helpers.max_rel(helpers.to_np(pkg["alpha"]), 1.0 - G["T"]) < 1e-6
    gc, gd, ga, gf = helpers.pixel_grads(cfg, device=DEV)
    loss = (pkg["render"] * gc).sum() + (pkg["depth"] * gd).sum() + (pkg["alpha"] * ga).sum() + (pkg["flow"] * gf).sum()
    loss.backward()
    checks = (("dL_dmeans3D", pc.get_xyz), ("dL_dopacity", pc.get_opacity), ("dL_dscales", pc.get_scaling),
              ("dL_dscales_t", pc.get_scaling_t), ("dL_drot", pc.get_rotation), ("dL_drot_r", pc.get_rotation_r),
              ("dL_dts", pc.get_t), ("dL_dsh", pc.get_features), ("dL_dmeans2D", pkg["viewspace_points"]))
    for gname, t in checks:
        ref = G["grad_" + gname]
        assert t.grad is not None, gname
        assert helpers.l2_rel(helpers.to_np(t.grad).reshape(ref.shape), ref) < 1e-4, gname
    # a loss on the image only (the reference's training loss, train.py:115-117): the unused outputs
    # contribute nothing -- same gradients as passing explicit zero upstream gradients
    pc2 = _Model(sc)
    pkg2 = render(cam.to(DEV), pc2, _Pipe(), bg)
    (pkg2["render"] * gc).sum().backward()
    fw = C.rasterize_gaussians(*helpers.fwd_args(st, sc, cfg))
    z = lambda t: torch.zeros_like(t)
    bw = C.rasterize_gaussians_backward(*helpers.bwd_args(st, sc, cfg, fw, (gc, z(gd), z(ga), z(gf))))
    assert helpers.l2_rel(helpers.to_np(pc2.get_xyz.grad), helpers.to_np(bw[3])) < 1e-5
    assert helpers.l2_rel(helpers.to_np(pc2.get_features.grad), helpers.to_np(bw[5])) < 1e-5


def test_render_python_preprocess_flags(C):
    """compute_cov3D_python / convert_SHs_python branches of render() (reference: __init__.py:73-81,98-111)
    against the all-CUDA path: same image up to the documented SH-direction quirk."""
    from gaussian_renderer import render, pyprep
    cfg, cam, sc, st = helpers.build("tiny", device=DEV)

    class M(_Model):
        def get_current_covariance_and_mean_offset(self, mod, timestamp):
            return pyprep.conditional_covariance_and_offset(torch.cat([self.get_scaling, self.get_scaling_t], 1), mod,
                                                            self.get_rotation, self.get_rotation_r, timestamp - self.get_t)

        def get_marginal_t(self, timestamp):
            return pyprep.marginal_t(torch.cat([self.get_scaling, self.get_scaling_t], 1), 1.0, self.get_rotation,
                                     self.get_rotation_r, self.get_t, timestamp)

    class P2(_Pipe):
        compute_cov3D_python = True
        convert_SHs_python = True

    bg = torch.zeros(3, device=DEV)
    a = render(cam.to(DEV), M(sc), _Pipe(), bg)
    b = render(cam.to(DEV), M(sc), P2(), bg)
    assert a["radii"].shape == b["radii"].shape
    agree = (a["radii"] > 0) == (b["radii"] > 0)
    assert float(agree.float().mean()) > 0.995
    assert helpers.psnr(helpers.to_np(a["render"]), helpers.to_np(b["render"])) > 35.0


def test_pack_unpack_rows_exchange_kernels(C):
    """csrc/exchange.cu (multi-GPU gradient exchange): gather of the union's rows into one flat buffer and the
    inverse scatter, bit-exact against torch indexing, vector (row % 16 B == 0) and scalar paths, ragged K."""
    g = torch.Generator(device=DEV).manual_seed(3)
    P = 10007
    tensors = [torch.randn(P, 3, device=DEV, generator=g), torch.randn(P, 48, 3, device=DEV, generator=g),
               torch.randn(P, 1, device=DEV, generator=g), torch.randn(P, 4, device=DEV, generator=g)]
    mask = torch.rand(P, device=DEV, generator=g) < 0.37
    idx = torch.nonzero(mask).squeeze(1)
    K = idx.numel()
    flat = C.pack_rows(tensors, idx)
    off = 0
    for t in tensors:
        w = t.numel() // P
        assert torch.equal(flat[off:off + K * w].view(K, w), t.view(P, w)[idx])
        off += (K * w + 3) // 4 * 4
    assert off == flat.numel()
    outs = [torch.zeros_like(t) for t in tensors]
    C.unpack_rows(flat, outs, idx)
    for o, t in zip(outs, tensors):
        assert torch.equal(o, t * mask.view(P, *([1] * (t.dim() - 1))))
    empty = torch.empty(0, dtype=torch.int64, device=DEV)
    assert C.pack_rows(tensors, empty).numel() == 0


# ---------------------------------------------------------------------------------------------------
# BASELINE config 4 ("lego" shape: 100k points in (-1.3, 1.3)^3, 800x800, batch of 2 views, 100 iterations):
# the optimisation loop of train.py:84-249 in miniature, once through this package's render(), once through the
# compiled reference rasterizer, same seeds -- the two loss curves must track each other.
# ---------------------------------------------------------------------------------------------------
from lego import lego_setup as _lego_setup, LegoModel as _LegoModel, lego_render as _lego_render  # noqa: E402


def test_cfg4_training_loop_tracks_reference(C):
    rec = helpers.ref_record("cfg4_loop")          # the reference's two loss curves (tools/ref_golden.py)
    P, W, H, iters, batch = 100_000, 800, 800, 100, 2
    cams, init, teacher = _lego_setup(P, W, H, seed=4)
    cams = [c.to(DEV) for c in cams]
    teacher_model = _LegoModel({k: v.to(DEV) for k, v in teacher.items()})
    with torch.no_grad():
        gts = [_lego_render(teacher_model, c, "ours").clone() for c in cams]   # synthetic ground truth
    for k, gt in enumerate(gts):
        assert helpers.digest(gt) == rec["gt%d" % k], k                       # the reference renders it bit for bit
    raw = {k: v.clone().to(DEV).requires_grad_(True) for k, v in init.items()}
    model = _LegoModel(raw)
    opt = torch.optim.Adam([{"params": [raw["xyz"]], "lr": 1.6e-4}, {"params": [raw["t"]], "lr": 1.6e-4},
                            {"params": [raw["sh"]], "lr": 2.5e-3}, {"params": [raw["op"]], "lr": 5e-2},
                            {"params": [raw["log_s"], raw["log_st"]], "lr": 5e-3},
                            {"params": [raw["rot"], raw["rot_r"]], "lr": 1e-3}], eps=1e-15)   # configs/dnerf/lego.yaml:36-44
    losses = []
    for it in range(iters):
        total = 0.0
        for b in range(batch):                      # sequential views, gradients accumulate (train.py:104-166)
            k = (it * batch + b) % len(cams)
            img = _lego_render(model, cams[k], "ours")
            loss = (img - gts[k]).abs().mean() / batch
            loss.backward()
            total += float(loss.detach())
        opt.step()
        opt.zero_grad(set_to_none=True)
        losses.append(total)
    ours, ref, ref2 = np.array(losses), rec["loss_ref"], rec["loss_ref_again"]
    assert np.isfinite(ours).all()
    assert ours[-1] < 0.8 * ours[0], "the loop is not optimising"            # it actually trains
    assert abs(ours[0] - ref[0]) <= 1e-6 * ref[0]                            # identical first loss (bit-exact forward)
    # Adam (eps 1e-15) turns every rounding-level gradient difference into a full-size step for near-zero
    # gradients, so trajectories separate chaotically -- the reference separates from ITSELF run to run (unordered
    # atomics).  The bar: our curve stays as close to the reference's as a second reference run does (x3), the early
    # iterations agree tightly, and the final loss agrees to 2 %.
    rel = np.abs(ours - ref) / ref
    self_rel = np.abs(ref2 - ref) / ref
    print("cfg4 loss curve: ours-vs-ref max %.3e mean %.3e | ref-vs-ref max %.3e mean %.3e | final %.5f vs %.5f"
          % (rel.max(), rel.mean(), self_rel.max(), self_rel.mean(), ours[-1], ref[-1]))
    assert rel[:10].max() < 1e-4, rel[:10]
    assert rel.mean() < 3 * self_rel.mean() + 1e-3 and rel.max() < 3 * self_rel.max() + 5e-3, (rel.max(), rel.mean(), self_rel.max(), self_rel.mean())
    tail = lambda c: float(c[-10:].mean())
    assert abs(tail(ours) - tail(ref)) < 3 * abs(tail(ref2) - tail(ref)) + 0.05 * tail(ref), (tail(ours), tail(ref), tail(ref2))
