#!/usr/bin/env python
"""Generates the committed golden vectors from the UNMODIFIED reference (compiled by oracle/build_ref.sh from
/root/reference/src, CPU/Embree path).  Run in the build container (where /root/reference exists):

    bash oracle/build_ref.sh && python tests/golden/make_golden.py

Each case renders a seeded synthetic scene (tests/scenes.py) through the host code in redner_b200/api.py with the
reference module as backend and stores the image and every gradient of loss = sum(img^2).
Cases with edge sampling whose samples cannot be reproduced sample-by-sample (secondary edges: the reference indexes
that stream by the rank of the pixel in its compacted active list, src/pathtracer.cpp:504-505) store the MEAN over
several seeds together with the standard error of that mean, for a statistical comparison.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402

import ref_loader  # noqa: E402
from parity_utils import (CASES, CORNERS, GBUFFER_CASES, GPU_CASES, REFSTREAM_CASES, SCREEN_CASES, STAT_CASES, pixel_sample, render_case,  # noqa: E402
                          render_corner, render_gbuffer, render_screen_gradient, render_stat_case)

OUT = os.path.dirname(os.path.abspath(__file__))


def main():
    ref = ref_loader.load()
    dev = torch.device("cpu")
    only = set(sys.argv[1:])  # optional: regenerate only the named cases
    for name, cfg in list(CASES.items()) + list(REFSTREAM_CASES.items()):
        if only and name not in only:
            continue
        img, grads = render_case(ref, dev, cfg, cfg["seed"])
        arrs = {"image": img.numpy()}
        for k, v in grads.items():
            arrs["grad." + k] = v.numpy()
        np.savez_compressed(os.path.join(OUT, name + ".npz"), **arrs)
        print(name, "image mean %.6f" % img.mean().item(), {k: float(v.norm()) for k, v in grads.items()})
    for name, cfg in GBUFFER_CASES.items():
        if only and name not in only:
            continue
        img = render_gbuffer(ref, dev, cfg)
        np.savez_compressed(os.path.join(OUT, name + ".npz"), image=img.numpy())
        print(name, tuple(img.shape), "mean %.6f" % img.mean().item())
    for name, cfg in SCREEN_CASES.items():
        if only and name not in only:
            continue
        img = render_screen_gradient(ref, dev, cfg)
        np.savez_compressed(os.path.join(OUT, name + ".npz"), image=img.numpy())
        print(name, tuple(img.shape), "norm %.6f" % img.norm().item())
    if not only or "c2_full_size_forward_blocks" in only:
        # the headline configuration itself (C2, 512 x 512 x 64 spp, forward): 8 x 8 block means of the reference's image
        cfg = dict(scene="shadow_blocker", res=512, spp=64, mb=1, sampler="sobol", edges=0)
        img, _ = render_case(ref, dev, cfg, 1, backward=False)
        np.savez_compressed(os.path.join(OUT, "c2_full_size_forward_blocks.npz"), blocks=img.numpy().reshape(64, 8, 64, 8, 3).mean((1, 3)))
        print("c2_full_size_forward_blocks", "mean %.6f" % img.mean().item())
    for name, cfg in STAT_CASES.items():
        if only and name not in only:
            continue
        acc = render_stat_case(ref, dev, name)
        arrs = {}
        for k, lst in acc.items():
            a = np.stack(lst)
            arrs["mean." + k] = a.mean(0)
            arrs["sem." + k] = a.std(0, ddof=1) / np.sqrt(len(lst))
            if cfg.get("test") == "ranks":  # per-seed values for the two-sample rank test (heavy-tailed estimators)
                arrs["samples." + k] = a
        np.savez_compressed(os.path.join(OUT, name + ".npz"), **arrs)
        print(name, {k: float(np.linalg.norm(v)) for k, v in arrs.items()})
    for name, cfg in GPU_CASES.items():
        if only and name not in only:
            continue
        img, grads = render_case(ref, dev, cfg, cfg["seed"], backward=name == "c2_shadow_blocker_128_sobol")
        img = img.numpy()
        arrs = {"pixels": img.reshape(-1, img.shape[-1])[pixel_sample(img.shape)], "image_max": np.float32(img.max())}
        arrs.update({"grad." + k: v.numpy() for k, v in grads.items()})
        np.savez_compressed(os.path.join(OUT, name + ".npz"), **arrs)
        print(name, "image mean %.6f" % img.mean(), sorted(arrs))
    for variant, chans, mb, edges, center in CORNERS:
        name = "corner_ball_" + variant
        if only and name not in only:
            continue
        img, grads = render_corner(ref, dev, variant, chans, mb, edges, center)
        np.savez_compressed(os.path.join(OUT, name + ".npz"), image=img, **{"grad." + k: v.numpy() for k, v in grads.items()})
        print(name, img.shape, sorted(grads))
    if not only or "fuzz_reference" in only:
        # the random scenes of tools/fuzz_emu.py that tests/test_device_code_cpu.py sweeps
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import fuzz_emu
        fuzz_emu.save_reference(ref, os.path.join(OUT, "fuzz_reference.npz"), 0, 80)
    if not only or "pyredner_envmap_tables" in only:
        save_pyredner_envmap_tables(os.path.join(OUT, "pyredner_envmap_tables.npz"))


def save_pyredner_envmap_tables(path):
    """The sampling tables, pdf normalisation and mip pyramid the reference's Python layer builds for one seeded environment map
    (pyredner/envmap.py, pyredner/texture.py), from the copy of pyredner that oracle/build_ref.sh places in oracle/_ref."""
    import types
    sys.path.insert(0, os.path.join(ROOT, "oracle", "_ref"))
    for name in ("skimage", "skimage.io", "skimage.transform", "imageio"):  # (image I/O the envmap code does not use)
        sys.modules.setdefault(name, types.ModuleType(name))
    sys.modules["skimage"].io = sys.modules["skimage.io"]
    sys.modules["skimage"].transform = sys.modules["skimage.transform"]
    sys.modules["redner"] = ref_loader.load()
    import pyredner
    import parity_utils as pu
    pyredner.set_use_gpu(False)
    sky, e2w = pu.envmap_table_inputs()
    a = pyredner.EnvironmentMap(sky, e2w)
    arrs = {"sample_cdf_xs": a.sample_cdf_xs.numpy(), "sample_cdf_ys": a.sample_cdf_ys.numpy(), "pdf_norm": np.float64(a.pdf_norm),
            "world_to_env": a.world_to_env.numpy()}
    arrs.update({"mip%d" % i: m.detach().numpy() for i, m in enumerate(a.values.mipmap)})
    np.savez_compressed(path, **arrs)
    print(os.path.basename(path), sorted(arrs))


if __name__ == "__main__":
    main()
