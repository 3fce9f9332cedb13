"""CPU suite, part 4: the drop-in claim.  Where oracle/build_ref.sh has placed the UNMODIFIED pyredner package in oracle/_ref, it
is imported on top of redner_b200/dropin/redner.py and its own RenderFunction marshals a scene all the
way into our C ABI (which then refuses to render without a GPU -- there is no CPU path)."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "oracle", "_ref")  # the unmodified pyredner and the reference's native module (oracle/build_ref.sh)

SCRIPT = r'''
import sys, types
sys.path.insert(0, %(ref)r)
sys.path.insert(0, %(dropin)r)  # (ahead of the reference's own native `redner` module next to pyredner)
for name in ("skimage", "skimage.io", "skimage.transform", "imageio"):
    sys.modules[name] = types.ModuleType(name)
sys.modules["skimage"].io = sys.modules["skimage.io"]
sys.modules["skimage"].transform = sys.modules["skimage.transform"]
import torch, pyredner, redner
assert redner.__file__.startswith(%(dropin)r), redner.__file__
pyredner.set_use_gpu(torch.cuda.is_available())
cam = pyredner.Camera(position=torch.tensor([0., 0., -5.]), look_at=torch.tensor([0., 0., 0.]), up=torch.tensor([0., 1., 0.]),
                      fov=torch.tensor([45.]), clip_near=1e-2, resolution=(16, 16))
dev = pyredner.get_device()
mat = pyredner.Material(diffuse_reflectance=torch.tensor([0.5, 0.5, 0.5], device=dev))
tri = pyredner.Shape(vertices=torch.tensor([[-2.0, 1.5, 0.3], [0.9, 1.2, -0.3], [-0.4, -1.4, 0.2]], device=dev),
                     indices=torch.tensor([[0, 1, 2]], dtype=torch.int32, device=dev), uvs=None, normals=None, material_id=0)
lgt = pyredner.Shape(vertices=torch.tensor([[-1., -1., -7.], [1., -1., -7.], [-1., 1., -7.], [1., 1., -7.]], device=dev),
                     indices=torch.tensor([[0, 1, 2], [1, 3, 2]], dtype=torch.int32, device=dev), uvs=None, normals=None, material_id=0)
scene = pyredner.Scene(cam, [tri, lgt], [mat], [pyredner.AreaLight(shape_id=1, intensity=torch.tensor([20., 20., 20.]))])
args = pyredner.RenderFunction.serialize_scene(scene=scene, num_samples=4, max_bounces=1)
try:
    img = pyredner.RenderFunction.apply(0, *args)
    print("RENDERED", float(img.mean()))
except RuntimeError as e:
    print("ABI-ERROR", e)
'''


@pytest.mark.skipif(not os.path.isdir(os.path.join(REF, "pyredner")), reason="oracle/_ref/pyredner not built")
def test_unmodified_pyredner_runs_on_the_dropin_module():
    code = SCRIPT % {"dropin": os.path.join(ROOT, "redner_b200", "dropin"), "ref": REF}
    out = subprocess.run([sys.executable, "-W", "ignore", "-c", code], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    last = out.stdout.strip().splitlines()[-1]
    # on a CPU-only machine the call must arrive at rb_scene_create and be refused loudly; on a GPU box it renders
    assert last.startswith("RENDERED") or ("ABI-ERROR" in last and "no CPU path" in last), last


def test_envmap_preprocessing_matches_pyredner():
    """api.EnvironmentMap builds the importance-sampling tables, pdf normalisation and mip pyramid that the reference's Python
    layer hands to the native EnvironmentMap (pyredner/envmap.py:36-61, pyredner/texture.py); the reference's tables for the
    same seeded map are stored in tests/golden/pyredner_envmap_tables.npz."""
    import numpy as np
    import torch
    import parity_utils as pu
    from redner_b200 import api
    g = pu.load_golden("pyredner_envmap_tables")
    sky, e2w = pu.envmap_table_inputs()
    b = api.EnvironmentMap(sky, e2w)
    assert np.array_equal(b.sample_cdf_xs.numpy(), g["sample_cdf_xs"]) and np.array_equal(b.sample_cdf_ys.numpy(), g["sample_cdf_ys"]), "sampling tables differ"
    assert abs(g["pdf_norm"] - b.pdf_norm) <= 1e-12 * abs(g["pdf_norm"]), (g["pdf_norm"], b.pdf_norm)
    assert np.array_equal(b.world_to_env.numpy(), g["world_to_env"])
    mips = sorted((k for k in g if k.startswith("mip")), key=lambda k: int(k[3:]))
    assert len(b.values.mipmap) == len(mips) and all(torch.allclose(x, torch.from_numpy(g[k]), atol=1e-7) for x, k in zip(b.values.mipmap, mips))


@pytest.mark.skipif(not os.path.isdir(os.path.join(REF, "pyredner")), reason="oracle/_ref/pyredner not built")
def test_unmodified_pyredner_gives_the_same_numbers_on_either_native_module(tmp_path):
    """The drop-in claim, numerically, without a GPU: the UNMODIFIED pyredner (its own serialize / unpack / forward / backward)
    renders and differentiates one scene twice -- on the reference's pybind module and on redner_b200/dropin/redner.py bound to
    the host build of the device headers (tools/cpu_emu, test infrastructure) -- and every number must agree."""
    import numpy as np
    import test_device_code_cpu as tdc
    emu = tdc._build()
    outs = {}
    for native in ("reference", emu):
        path = str(tmp_path / ("ref.npz" if native == "reference" else "ours.npz"))
        r = subprocess.run([sys.executable, "-W", "ignore", os.path.join(ROOT, "tests", "dropin_script.py"), native, path, REF, "cpu"], capture_output=True, text=True,
                           timeout=600)
        assert r.returncode == 0 and "DONE" in r.stdout, r.stderr[-3000:]
        outs[native] = dict(np.load(path))
    a, b = outs["reference"], outs[emu]
    rel = lambda x, y: float(np.linalg.norm(x.astype(np.float64) - y) / max(np.linalg.norm(y), 1e-30))  # noqa: E731
    for k in a:
        if np.linalg.norm(a[k]) < 1e-4:  # (e.g. the roughness of a surface no specular path reaches)
            continue
        tol = 1e-5 if k.endswith("image") else (2e-3 if k.startswith(("edge_", "opt_")) else 2e-4)  # edge rays graze silhouettes: a hit may flip
        assert rel(b[k], a[k]) < tol, (k, rel(b[k], a[k]))
