#!/usr/bin/env python3
"""Writes tests/golden/ref_*.npz: compact records of the compiled, unmodified reference rasterizer (oracle/_ref,
built by oracle/build_ref.py) for the GPU tests that compare with it at sizes too large to store whole
(tests/helpers.py: digest, grad_record).  Needs a GPU and oracle/_ref/ref_rasterizer.so.

  full_<name>     forward digests (radii, images, out_means3D, cov3D of the visible Gaussians, the reference's tile
                  lists) and the 12 gradients over REF_RERUNS backward reruns, upstream gradients of every image
  colour_<name>   the 12 gradients with only the colour image carrying an upstream gradient
  raw_cfg3        cfg3 through the reference's torch prologue over raw parameters: a pixel sample of the image and
                  the gradients of the raw leaves over 3 runs
  cfg4_loop       the lego-shape training loop: digests of the ground-truth renders, two reference loss curves

Usage: python tools/ref_golden.py --out DIR [--only full_mid,...]
"""
import argparse
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in ("4d-gaussian-splatting_b200", "oracle", "tests"):
    sys.path.insert(0, os.path.join(ROOT, p))

import helpers  # noqa: E402
import oracle_py  # noqa: E402

DEV = "cuda:0"
REF_RERUNS = 8
FULL = ["mid", "mid_rotcam", "mid_dur10", "mid_smod2", "cfg5", "cfg2", "cfg3"]
COLOUR = ["small", "ragged", "negfov", "rotcam", "n3v", "mid", "mid_dur10", "cfg5", "cfg2", "cfg3"]


def grads_record(reruns):
    return {gname: helpers.grad_record([r[k] for r in reruns], seed=1000 + k) for k, gname in enumerate(helpers.GRAD_NAMES)}


def full(name):
    ref = oracle_py.ref_module()
    cfg, cam, sc, st = helpers.build(name, device=DEV)
    W, H = cfg["W"], cfg["H"]
    grads = helpers.pixel_grads(cfg, device=DEV)
    rf = ref.rasterize_gaussians(*helpers.fwd_args(st, sc, cfg))
    reruns = [ref.rasterize_gaussians_backward(*helpers.bwd_args(st, sc, cfg, rf, grads)) for _ in range(REF_RERUNS)]
    torch.cuda.synchronize()
    ri = oracle_py.ref_image_views(rf[8], W * H)
    n_tiles = ((W + 15) // 16) * ((H + 15) // 16)
    lists = dict(point_list=helpers.to_np(oracle_py.ref_binning_point_list(rf[7], rf[0])),
                 ranges=helpers.to_np(ri["ranges"][:n_tiles]), n_contrib=helpers.to_np(ri["n_contrib"]), num_rendered=int(rf[0]))
    digests = helpers.list_digests(lists)
    for i, key in ((5, "radii"), (1, "color"), (2, "flow"), (3, "depth"), (4, "T"), (10, "out_means3D")):
        digests[key] = helpers.digest(rf[i])
    digests["cov3D"] = helpers.digest(rf[9][rf[5] > 0])
    return dict(grads_record(reruns), digests=helpers.pack_digests(digests))


def colour(name):
    ref = oracle_py.ref_module()
    cfg, cam, sc, st = helpers.build(name, device=DEV)
    gc, gd, ga, gf = helpers.pixel_grads(cfg, device=DEV)
    rf = ref.rasterize_gaussians(*helpers.fwd_args(st, sc, cfg))
    zeros = (gc, 0 * gd, 0 * ga, 0 * gf)
    reruns = [ref.rasterize_gaussians_backward(*helpers.bwd_args(st, sc, cfg, rf, zeros)) for _ in range(REF_RERUNS)]
    torch.cuda.synchronize()
    return dict(grads_record(reruns), digests=helpers.pack_digests({}))


def raw_cfg3():
    import ref_api
    from raw_model import RawModel
    cfg, cam, sc, st = helpers.build("cfg3", device=DEV)
    g = torch.Generator().manual_seed(77)
    G = torch.randn(3, cfg["H"], cfg["W"], generator=g).to(DEV)

    def ref_run():
        R = RawModel(sc, seed=2, requires_grad=True)
        m2 = torch.zeros_like(R._xyz, requires_grad=True)
        out = ref_api.rasterize(st, R.get_xyz, m2, R.get_opacity, R.get_features, torch.zeros(sc.P, 2, device=DEV), R.get_t,
                                R.get_scaling, R.get_scaling_t, R.get_rotation, R.get_rotation_r)
        (out[0] * G).sum().backward()
        return R, out[0].detach()

    runs = [ref_run() for _ in range(3)]
    pix = torch.sort(torch.randperm(cfg["H"] * cfg["W"], generator=torch.Generator().manual_seed(78))[:1024]).values
    rec = {"pixels": pix.numpy().astype(np.int32), "image": helpers.to_np(runs[0][1].reshape(3, -1)[:, pix.to(DEV)]),
           "digests": helpers.pack_digests({})}
    for i, k in enumerate(runs[0][0].leaves()):
        rec[k] = helpers.grad_record([r[0].leaves()[k].grad for r in runs], seed=2000 + i)
    return rec


def cfg4_loop():
    """The reference arm of tests/test_gpu_parity.py::test_cfg4_training_loop_tracks_reference, twice."""
    from lego import lego_setup, LegoModel, lego_render
    P, W, H, iters, batch = 100_000, 800, 800, 100, 2
    cams, init, teacher = lego_setup(P, W, H, seed=4)
    cams = [c.to(DEV) for c in cams]
    teacher_model = LegoModel({k: v.to(DEV) for k, v in teacher.items()})
    with torch.no_grad():
        gts = [lego_render(teacher_model, c, "ref").clone() for c in cams]
    rec = {"digests": helpers.pack_digests({"gt%d" % k: helpers.digest(gt) for k, gt in enumerate(gts)})}
    for label in ("loss_ref", "loss_ref_again"):
        raw = {k: v.clone().to(DEV).requires_grad_(True) for k, v in init.items()}
        model = LegoModel(raw)
        opt = torch.optim.Adam([{"params": [raw["xyz"]], "lr": 1.6e-4}, {"params": [raw["t"]], "lr": 1.6e-4},
                                {"params": [raw["sh"]], "lr": 2.5e-3}, {"params": [raw["op"]], "lr": 5e-2},
                                {"params": [raw["log_s"], raw["log_st"]], "lr": 5e-3},
                                {"params": [raw["rot"], raw["rot_r"]], "lr": 1e-3}], eps=1e-15)
        losses = []
        for it in range(iters):
            total = 0.0
            for b in range(batch):
                k = (it * batch + b) % len(cams)
                loss = (lego_render(model, cams[k], "ref") - gts[k]).abs().mean() / batch
                loss.backward()
                total += float(loss.detach())
            opt.step()
            opt.zero_grad(set_to_none=True)
            losses.append(total)
        rec[label] = np.array(losses)
    return rec


def python_call(out):
    """CPU, needs the reference's source tree: its own gaussian_renderer/diff_gaussian_rasterization.py (everything after
    the `_C = load(...)` JIT preamble) run with `_C` replaced by a recorder.  Writes DIR/ref_python_call.json: the
    settings' field names and the kind of each positional argument it passes to _C.rasterize_gaussians -- an input
    tensor by name, an empty placeholder, or a Python scalar with its value."""
    import json
    from typing import NamedTuple
    import build_ref
    ref_file = os.path.join(build_ref.REF, "gaussian_renderer", "diff_gaussian_rasterization.py")
    src = open(ref_file).read()

    class Recorded(Exception):
        pass

    calls = []

    class Recorder:
        def rasterize_gaussians(self, *args):
            calls.append(args)
            raise Recorded

    ns = {"torch": torch, "nn": torch.nn, "_C": Recorder(), "__name__": "ref_dgr_recorded", "NamedTuple": NamedTuple}
    exec(compile(src[src.index("def cpu_deep_copy_tuple"):], ref_file, "exec"), ns)
    cfg, cam, sc, st = helpers.build("tiny")
    settings = ns["GaussianRasterizationSettings"](**st)
    inputs = dict(means3D=sc.means3D, means2D=torch.zeros_like(sc.means3D), opacities=sc.opacities, shs=sc.shs,
                  flow_2d=sc.flow_2d, ts=sc.ts, scales=sc.scales, scales_t=sc.scales_t, rotations=sc.rotations,
                  rotations_r=sc.rotations_r)
    try:
        ns["GaussianRasterizer"](settings)(**inputs)
    except Recorded:
        pass
    named = {id(v): k for k, v in inputs.items()}
    named.update({id(st[f]): "settings." + f for f in settings._fields if isinstance(st[f], torch.Tensor)})
    desc = []
    for a in calls[0]:
        if isinstance(a, torch.Tensor):
            assert id(a) in named or a.numel() == 0, a.shape
            desc.append({"tensor": named.get(id(a), "empty")})
        else:
            desc.append({type(a).__name__: a})
    os.makedirs(out, exist_ok=True)
    with open(os.path.join(out, "ref_python_call.json"), "w") as f:
        json.dump({"fields": list(settings._fields), "rasterize_gaussians": desc}, f, indent=1)
        f.write("\n")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--only", default="")
    ap.add_argument("--python-call", action="store_true", help="only ref_python_call.json (CPU, reference sources)")
    args = ap.parse_args()
    if args.python_call:
        return python_call(args.out)
    assert torch.cuda.is_available() and oracle_py.ref_available(), "needs a GPU and oracle/_ref/ref_rasterizer.so"
    jobs = [("full_" + n, full, n) for n in FULL] + [("colour_" + n, colour, n) for n in COLOUR] + \
           [("raw_cfg3", raw_cfg3, None), ("cfg4_loop", cfg4_loop, None)]
    only = set(filter(None, args.only.split(",")))
    os.makedirs(args.out, exist_ok=True)
    for tag, fn, arg in jobs:
        if only and tag not in only:
            continue
        rec = fn(arg) if arg is not None else fn()
        path = os.path.join(args.out, "ref_%s.npz" % tag)
        np.savez_compressed(path, **rec)
        print("%-22s %7d bytes" % (tag, os.path.getsize(path)), flush=True)
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
