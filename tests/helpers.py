"""Shared helpers of the parity tests: seeded configurations, runners for the three
implementations (CUDA path through the extension, CPU oracle, compiled reference) and the
comparison metrics (SURVEY.md section 8d)."""
import hashlib
import os

import numpy as np
import torch

from fdgs import synth
import oracle_py

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")

# name -> synthetic configuration.  The ones with a golden_<name>.npz were run through the UNMODIFIED
# reference kernels on a B200 (tools/first_light.py --golden, see tests/golden/README.md).
CONFIGS = {
    "tiny": dict(P=2000, W=128, H=96, seed=11),
    "small": dict(P=10000, W=256, H=256, seed=1235),
    "flowbg": dict(P=3000, W=160, H=112, seed=77, flow=True, bg=(0.3, 0.6, 0.1)),
    "negfov": dict(P=3000, W=160, H=112, seed=78, negative_fov=True, flow=True),
    "ragged": dict(P=1500, W=101, H=67, seed=5),            # image not a multiple of the 16x16 tile
    "sh3d": dict(P=3000, W=160, H=112, seed=79, force_sh_3d=True),
    "dim3": dict(P=3000, W=160, H=112, seed=80, gaussian_dim=3, rot_4d=False),
    "norot4d": dict(P=3000, W=160, H=112, seed=81, gaussian_dim=4, rot_4d=False),
    "deg1": dict(P=3000, W=160, H=112, seed=82, sh_degree=1, sh_degree_t=0, M=48),
    "m16": dict(P=3000, W=160, H=112, seed=83, sh_degree=3, sh_degree_t=0, M=16),
    "prefilter": dict(P=3000, W=160, H=112, seed=84, prefilter_var=0.01),
    # --- inputs the first golden set never exercised (VERDICT r1, weak #1) ---
    # N3V-style time axis: duration 10, timestamps off 0.5 -> the double-precision Fourier angle of the 4D SH
    "dur10": dict(P=3000, W=160, H=112, seed=85, time_duration=10.0, timestamp=3.7, scale_t_mean=1.2),
    # densification previews render with scaling_modifier != 1 (reference: gaussian_renderer/__init__.py:19,39)
    "smod05": dict(P=3000, W=160, H=112, seed=86, scale_modifier=0.5),
    "smod2": dict(P=3000, W=160, H=112, seed=87, scale_modifier=2.0),
    # rotated + translated camera: non-identity view matrix, campos != 0 (every SH direction, the EWA Jacobian)
    "rotcam": dict(P=3000, W=160, H=112, seed=88, pose=(25.0, -10.0, 5.0, 0.7, -0.4, 1.2), flow=True, bg=(0.2, 0.1, 0.4)),
    # flame_steak shape in miniature: duration [0,10], negative FoV (quirk 7), posed camera, all at once
    "n3v": dict(P=3000, W=160, H=112, seed=89, time_duration=10.0, timestamp=6.3, scale_t_mean=1.2, negative_fov=True,
                pose=(-15.0, 8.0, -3.0, -0.5, 0.3, 0.8)),
    "deg1m4": dict(P=3000, W=160, H=112, seed=90, sh_degree=1, sh_degree_t=0, M=4),   # row shorter than a 16-block
    "mid": dict(P=100000, W=640, H=480, seed=1236),
    "mid_rotcam": dict(P=100000, W=640, H=480, seed=1238, pose=(25.0, -10.0, 5.0, 0.7, -0.4, 1.2)),
    "mid_dur10": dict(P=100000, W=640, H=480, seed=1239, time_duration=10.0, timestamp=3.7, scale_t_mean=1.2),
    "mid_smod2": dict(P=100000, W=640, H=480, seed=1240, scale_modifier=2.0),
    "q250k": dict(P=250000, W=478, H=358, seed=1237),          # 1/8-scale replica of cfg3 (same density)
    # BASELINE config 5 (N3V flame_steak shape): 300k Gaussians, duration [0,10], 1352x1014, posed N3V-style camera
    "cfg5": dict(P=300000, W=1352, H=1014, seed=1241, time_duration=10.0, timestamp=4.3, scale_t_mean=1.2,
                 pose=(10.0, -5.0, 0.0, 0.3, -0.2, 0.5)),
    "cfg2": dict(P=500000, W=1352, H=1014, seed=1236),
    "cfg3": dict(P=2000000, W=1352, H=1014, seed=1237),
}

GRAD_NAMES = ["dL_dmeans2D", "dL_dcolors", "dL_dopacity", "dL_dmeans3D", "dL_dcov3D", "dL_dsh", "dL_dflows", "dL_dts",
              "dL_dscales", "dL_dscales_t", "dL_drot", "dL_drot_r"]
# same order, names used by oracle_py.backward
ORACLE_GRAD_KEYS = ["dL_dmeans2D", "dL_dcolors", "dL_dopacity", "dL_dmeans3D", "dL_dcov3D", "dL_dsh", "dL_dflows", "dL_dts",
                    "dL_dscales", "dL_dscales_t", "dL_drotations", "dL_drotations_r"]


def build(name_or_cfg, device="cpu"):
    cfg = CONFIGS[name_or_cfg] if isinstance(name_or_cfg, str) else name_or_cfg
    R = T = None
    if cfg.get("pose") is not None:
        R, T = synth.pose_from_euler(*cfg["pose"])
    cam = synth.make_camera(cfg["W"], cfg["H"], timestamp=cfg.get("timestamp", 0.5),
                            negative_fov=cfg.get("negative_fov", False), R=R, T=T)
    sc = synth.make_scene(cfg["P"], cam, cfg["seed"], flow=cfg.get("flow", False), M=cfg.get("M", 48),
                          sh_degree=cfg.get("sh_degree", 3), sh_degree_t=cfg.get("sh_degree_t", 2),
                          rot_4d=cfg.get("rot_4d", True), gaussian_dim=cfg.get("gaussian_dim", 4),
                          force_sh_3d=cfg.get("force_sh_3d", False), time_duration=cfg.get("time_duration", 1.0),
                          scale_t_mean=cfg.get("scale_t_mean", 0.15))
    bg = torch.tensor(cfg.get("bg", (0.0, 0.0, 0.0)), dtype=torch.float32)
    st = synth.raster_settings(cam, sc, bg=bg, scale_modifier=cfg.get("scale_modifier", 1.0), device=device)
    return cfg, cam, sc.to(device), st


def pixel_grads(cfg, device="cpu"):
    g = torch.Generator().manual_seed(cfg["seed"] + 999)
    H, W = cfg["H"], cfg["W"]
    gc = torch.randn(3, H, W, generator=g)
    gd = 0.1 * torch.randn(1, H, W, generator=g)
    ga = 0.1 * torch.randn(1, H, W, generator=g)
    gf = 0.1 * torch.randn(2, H, W, generator=g)
    return tuple(t.to(device) for t in (gc, gd, ga, gf))


def _opt(t, sc, cond=True):
    return t if cond else torch.Tensor([])


def fwd_args(st, sc, cfg):
    """Positional arguments of _C.rasterize_gaussians (reference: diff_gaussian_rasterization.py:88-119)."""
    e = torch.Tensor([])
    four_d = sc.gaussian_dim == 4
    return (st["bg"], sc.means3D, e, sc.flow_2d, sc.opacities, sc.ts if four_d else e, sc.scales,
            sc.scales_t if four_d else e, sc.rotations, sc.rotations_r if sc.rot_4d else e, st["scale_modifier"], e,
            cfg.get("prefilter_var", -1.0), st["viewmatrix"], st["projmatrix"], st["tanfovx"], st["tanfovy"],
            st["image_height"], st["image_width"], sc.shs, st["sh_degree"], st["sh_degree_t"], st["campos"],
            st["timestamp"], st["time_duration"], st["rot_4d"], st["gaussian_dim"], st["force_sh_3d"],
            st["prefiltered"], st["debug"])


def bwd_args(st, sc, cfg, fw, grads):
    e = torch.Tensor([])
    four_d = sc.gaussian_dim == 4
    (num_rendered, color, flow, depth, T, radii, geom, binning, img, covs, out_means3D) = fw
    gc, gd, ga, gf = grads
    return (st["bg"], sc.means3D, out_means3D, radii, e, sc.flow_2d, sc.opacities, sc.ts if four_d else e, sc.scales,
            sc.scales_t if four_d else e, sc.rotations, sc.rotations_r if sc.rot_4d else e, st["scale_modifier"], e,
            cfg.get("prefilter_var", -1.0), st["viewmatrix"], st["projmatrix"], st["tanfovx"], st["tanfovy"], gc, gd, ga,
            gf, sc.shs, st["sh_degree"], st["sh_degree_t"], st["campos"], st["timestamp"], st["time_duration"],
            st["rot_4d"], st["gaussian_dim"], st["force_sh_3d"], geom, num_rendered, binning, img, st["debug"])


def oracle_inputs(st, sc, cfg):
    four_d = sc.gaussian_dim == 4
    return oracle_py.OracleInputs(st, sc.means3D, sc.opacities, shs=sc.shs, flow_2d=sc.flow_2d,
                                  ts=sc.ts if four_d else None, scales=sc.scales,
                                  scales_t=sc.scales_t if four_d else None, rotations=sc.rotations,
                                  rotations_r=sc.rotations_r if sc.rot_4d else None,
                                  prefilter_var=cfg.get("prefilter_var", -1.0))


def bitdiff(a, b):
    """number of elements whose bit patterns differ"""
    a = np.ascontiguousarray(a)
    b = np.ascontiguousarray(b)
    assert a.shape == b.shape, (a.shape, b.shape)
    if a.dtype.kind == "f":
        return int((a.view(np.int32) != b.view(np.int32)).sum())
    return int((a.astype(np.int64) != b.astype(np.int64)).sum())


def max_rel(a, b):
    """max-norm relative error ||a-b||_inf / ||b||_inf  (SURVEY.md section 8d)"""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    n = np.abs(b).max() if b.size else 0.0
    d = np.abs(a - b).max() if b.size else 0.0
    return d / n if n > 0 else d


def l2_rel(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    n = np.sqrt((b * b).sum())
    return np.sqrt(((a - b) ** 2).sum()) / n if n > 0 else np.sqrt(((a - b) ** 2).sum())


def psnr(a, b):
    mse = float(((np.asarray(a, np.float64) - np.asarray(b, np.float64)) ** 2).mean())
    return 200.0 if mse == 0 else 10.0 * np.log10(1.0 / mse)


def golden(name):
    path = os.path.join(GOLDEN_DIR, "golden_%s.npz" % name)
    return np.load(path) if os.path.exists(path) else None


# ---- compact records of the reference at sizes too large to store whole (tests/golden/ref_*.npz, written by
# tools/ref_golden.py from the compiled reference).  Bit-exact outputs are kept as SHA-256 digests; gradients as the
# mean of the reference's reruns on a seeded sample of rows (the largest rows plus random ones) with the reference's
# run-to-run spread on that sample and over the whole tensor, and the norm of the whole mean tensor.
SAMPLE_TOP, SAMPLE_RANDOM, SAMPLE_COLS = 16, 32, 12
GRAD_STATS = ("nm_full", "l2n_full", "l2max_full", "l2n", "l2max", "mxn", "rmed")
GRAD_EMPTY, GRAD_ZERO = -1.0, 0.0          # one-element records: the reference returned an empty / an all-zero tensor


def ref_record(name):
    """tests/golden/ref_<name>.npz as a dict: every digest by its name (a str), every other array as stored."""
    with np.load(os.path.join(GOLDEN_DIR, "ref_%s.npz" % name)) as z:
        rec = {k: z[k] for k in z.files if k != "digests"}
        rec.update(s.decode().split("=", 1) for s in z["digests"])
    return rec


def pack_digests(d):
    return np.array(["%s=%s" % kv for kv in d.items()], dtype="S")


def digest(t):
    """SHA-256 of a tensor's values: floats by their fp32 bit patterns, integers widened to int64."""
    a = np.ascontiguousarray(to_np(t) if hasattr(t, "detach") else np.asarray(t))
    if a.dtype.kind == "f":
        assert a.dtype == np.float32, a.dtype
    else:
        a = a.astype(np.int64)
    return "%s:%s" % (a.size, hashlib.sha256(a.reshape(-1).tobytes()).hexdigest())


def list_digests(lists):
    """Digests of the tile lists of check_tile_lists's dict layout."""
    return dict(point_list=digest(np.asarray(lists["point_list"]).reshape(-1)),
                ranges=digest(np.asarray(lists["ranges"]).reshape(-1, 2)),
                n_contrib=digest(np.asarray(lists["n_contrib"]).reshape(-1)), num_rendered=str(int(lists["num_rendered"])))


def median_row_err(x, m):
    d = (x - m).norm(dim=1)
    n = m.norm(dim=1)
    keep = n > 0
    return (d[keep] / n[keep]).median().item() if bool(keep.any()) else 0.0


def pack_grad(rows, cols, mean, stats):
    """One float32 array: [len(rows), len(cols), GRAD_STATS..., rows, cols, mean (rows x cols)]; indices < 2^24."""
    assert len(rows) == 0 or int(np.max(rows)) < (1 << 24)
    return np.concatenate([[len(rows), len(cols)], stats, rows, cols, np.asarray(mean).reshape(-1)]).astype(np.float32)


def grad_record(runs, seed):
    """Record of K reference reruns of one gradient tensor (list of K tensors [P, ...]) for grad_sample."""
    if runs[0].numel() == 0:
        return np.array([GRAD_EMPTY], np.float32)
    P = runs[0].shape[0]
    flat = lambda r: r.detach().reshape(P, -1).double()
    m = sum(flat(r) for r in runs) / len(runs)
    nm = m.norm().item()
    if nm == 0.0:
        return np.array([GRAD_ZERO], np.float32)
    rel = [(flat(r) - m).norm().item() / nm for r in runs]
    n = m.norm(dim=1)
    nz = torch.nonzero(n > 0).squeeze(1)
    g = torch.Generator().manual_seed(seed)
    pick = torch.randperm(nz.numel(), generator=g)[:SAMPLE_RANDOM].to(nz.device)
    rows = torch.unique(torch.cat([torch.topk(n, min(SAMPLE_TOP, nz.numel())).indices, nz[pick]]))
    live = torch.nonzero(m.abs().amax(0) > 0).squeeze(1)
    cols = live[torch.sort(torch.randperm(live.numel(), generator=g)[:SAMPLE_COLS]).values.to(live.device)]
    S = torch.stack([flat(r)[rows][:, cols] for r in runs]).cpu()
    rows, cols = rows.cpu(), cols.cpu()
    del m, n
    ms = S.mean(0)
    nms, scs = ms.norm().item(), ms.abs().max().item()
    rels = [(s - ms).norm().item() / nms for s in S]
    stats = [nm, float(np.sqrt(np.mean(np.square(rel)))), max(rel), float(np.sqrt(np.mean(np.square(rels)))), max(rels),
             max((s - ms).abs().max().item() for s in S) / scs, max(median_row_err(s, ms) for s in S)]
    return pack_grad(rows.numpy(), cols.numpy(), ms.numpy(), stats)


def grad_sample(p, a):
    """p: a grad_record (neither GRAD_EMPTY nor GRAD_ZERO); a: our gradient tensor.  Returns (ours on the record's
    sample, the reference mean there, | |ours| / |reference mean| - 1 | over the whole tensor, the statistics by name)."""
    nr, nc = int(p[0]), int(p[1])
    st = dict(zip(GRAD_STATS, p[2:2 + len(GRAD_STATS)].astype(np.float64).tolist()))
    o = 2 + len(GRAD_STATS)
    rows = torch.from_numpy(p[o:o + nr].astype(np.int64))
    cols = torch.from_numpy(p[o + nr:o + nr + nc].astype(np.int64))
    mean = torch.from_numpy(p[o + nr + nc:].astype(np.float64)).reshape(nr, nc)
    a = a.detach().double().reshape(a.shape[0], -1)
    s = a[rows.to(a.device)][:, cols.to(a.device)].cpu()
    return s, mean, abs(a.norm().item() / st["nm_full"] - 1.0), st


def to_np(t):
    return t.detach().cpu().numpy()


def check_tile_lists(ours, ref, W, H, mode):
    """Compare the private tile lists with the reference's.  ours / ref: dicts of numpy arrays
    point_list [R], ranges [tiles, 2], n_contrib [H*W] (and num_rendered).

    mode 0 (fdgs_set_tile_cull(0)): bit-identical.
    mode 1 (default): every tile's list is the reference's list with some instances REMOVED (same order), and every
    pixel's last contributor is the same Gaussian -- n_contrib itself counts positions of the shorter list.  That the
    removed instances blend nowhere is what the bit-identical images of the same tests prove."""
    op, orr, on = (np.asarray(ours[k]) for k in ("point_list", "ranges", "n_contrib"))
    rp, rr, rn = (np.asarray(ref[k]) for k in ("point_list", "ranges", "n_contrib"))
    orr, rr = orr.reshape(-1, 2).astype(np.int64), rr.reshape(-1, 2).astype(np.int64)
    on, rn = on.reshape(-1).astype(np.int64), rn.reshape(-1).astype(np.int64)
    if mode == 0:
        assert int(ours["num_rendered"]) == int(ref["num_rendered"])
        assert bitdiff(op, rp) == 0 and bitdiff(orr, rr) == 0 and bitdiff(on, rn) == 0
        return
    assert int(ours["num_rendered"]) <= int(ref["num_rendered"])
    assert orr.shape == rr.shape
    T = orr.shape[0]
    olen, rlen = orr[:, 1] - orr[:, 0], rr[:, 1] - rr[:, 0]
    assert int(olen.sum()) == int(ours["num_rendered"]) == len(op)
    assert (olen <= rlen).all()
    # (tile, gaussian) keys in list order; ours must equal the reference's filtered to the keys ours holds
    otile = np.repeat(np.arange(T, dtype=np.int64), olen)
    rtile = np.repeat(np.arange(T, dtype=np.int64), rlen)
    # lists are stored tile after tile in both implementations; rebuild that order explicitly from the ranges
    oidx = np.concatenate([np.arange(a, b) for a, b in orr if b > a]) if len(op) else np.zeros(0, np.int64)
    ridx = np.concatenate([np.arange(a, b) for a, b in rr if b > a]) if len(rp) else np.zeros(0, np.int64)
    okey = (otile << 32) | op[oidx].astype(np.int64)
    rkey = (rtile << 32) | rp[ridx].astype(np.int64)
    keep = np.isin(rkey, okey)
    assert int(keep.sum()) == len(okey), "our lists hold an instance the reference's do not"
    assert (rkey[keep] == okey).all(), "order inside a tile differs from the reference"
    # last contributor of every pixel: the same Gaussian
    gx = (W + 15) // 16
    ys, xs = np.divmod(np.arange(W * H, dtype=np.int64), W)
    tile = (ys // 16) * gx + xs // 16
    assert ((on > 0) == (rn > 0)).all()
    nz = on > 0
    g_ours = op[orr[tile[nz], 0] + on[nz] - 1]
    g_ref = rp[rr[tile[nz], 0] + rn[nz] - 1]
    assert (g_ours == g_ref).all(), "a pixel's last contributor differs"
