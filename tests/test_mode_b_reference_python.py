"""CPU: INTEGRATION.md mode B -- the reference's OWN gaussian_renderer/diff_gaussian_rasterization.py (classes and
autograd function, lines after its JIT-load preamble) driving this repo's extension as its `_C`.  What that layer
passes is recorded in tests/golden/ref_python_call.json (tools/ref_golden.py --python-call ran it with a recording
`_C`): the settings' field names and the 30 positional arguments of `_C.rasterize_gaussians` in the reference's order
and types.  The test replays that call on the extension; without a GPU it can only go as far as the extension's first
device check, and that point is reached only if pybind accepted the reference's argument list (a signature mismatch
raises TypeError first)."""
import json
import os

import pytest

import helpers


def test_reference_python_layer_binds_to_our_extension():
    import fdgs
    from gaussian_renderer import GaussianRasterizationSettings as Ours
    with open(os.path.join(helpers.GOLDEN_DIR, "ref_python_call.json")) as f:
        rec = json.load(f)
    assert list(Ours._fields) == rec["fields"]
    cfg, cam, sc, st = helpers.build("tiny")
    import torch
    inputs = dict(means3D=sc.means3D, opacities=sc.opacities, shs=sc.shs, flow_2d=sc.flow_2d, ts=sc.ts, scales=sc.scales,
                  scales_t=sc.scales_t, rotations=sc.rotations, rotations_r=sc.rotations_r, empty=torch.Tensor([]))
    inputs.update({"settings." + k: v for k, v in st.items()})
    casts = {"float": float, "int": int, "bool": bool}
    args = []
    for a in rec["rasterize_gaussians"]:
        (kind, v), = a.items()
        args.append(inputs[v] if kind == "tensor" else casts[kind](v))
    assert len(args) == 30
    # full call: the reference's argument list -> our shim.  On CPU tensors our shim stops at its device check -- after
    # pybind matched the reference's argument list.
    with pytest.raises(RuntimeError, match="means3D must be a CUDA tensor"):
        fdgs.ext().rasterize_gaussians(*args)
    assert hasattr(fdgs.ext(), "rasterize_gaussians_backward") and hasattr(fdgs.ext(), "mark_visible")
