"""Randomised parity sweep on a machine WITHOUT a GPU: random scenes / cameras / materials / options are rendered and
differentiated by (a) the compiled unmodified reference (oracle/_ref) and (b) the device headers compiled with g++
(tools/cpu_emu), through the same host code; every image and gradient is compared.

The reference's outputs come from the compiled reference (oracle/_ref) or, with --golden, from a file written by
save_reference (tests/golden/fuzz_reference.npz holds seeds 0 - 79).  Combinations on which the reference
itself corrupts its heap are not generated (no radiance channel with bounces, generic texture with primary edges:
DESIGN.md section 4); with secondary edge sampling (sample streams not reproducible one-to-one) or textured scenes under
primary edge sampling (stale footprints in the reference) only the non-geometric gradients are compared.

usage: python tools/fuzz_emu.py <emulator.so> <first seed> <count> [--verbose] [--golden <reference outputs.npz>]
"""
import ctypes
import math
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "oracle")):
    sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402


NO_IMAGE_TEXTURES = False  # (debugging aid: constant reflectances only)


def make_case(seed):
    from redner_b200 import api
    import scenes
    r = np.random.RandomState(seed)
    g = torch.Generator().manual_seed(seed)
    dev = torch.device("cpu")

    def T(x, grad=False, dt=torch.float32):
        t = torch.tensor(x, dtype=dt) if not isinstance(x, torch.Tensor) else x.to(dt)
        return t.requires_grad_(True) if grad else t

    def coin(p=0.5):
        return bool(r.rand() < p)
    cfg = {}
    # options first: they restrict what the scene may contain
    generic = coin(0.15)
    mb = int(r.randint(0, 4))
    chans = None
    if coin(0.3):
        names = ["alpha", "depth", "position", "geometry_normal", "shading_normal", "uv", "barycentric_coordinates", "diffuse_reflectance",
                 "specular_reflectance", "roughness", "vertex_color", "shape_id", "triangle_id", "material_id"] + (["generic_texture"] if generic else [])
        pick = list(r.choice(names, size=int(r.randint(1, 5)), replace=False))
        if coin(0.7):
            chans = ["radiance"] + pick
        else:
            chans, mb = pick, 0  # (no radiance channel: the reference is only safe without bounces)
    if chans is None:
        mb = max(mb, 1)  # (radiance alone without a bounce is black unless a lamp is in view)
    edges = coin(0.5) and not generic
    sampler = str(r.choice(["sobol", "independent"]))
    if sampler == "independent":
        # PCG streams: the reference stops a sample's bounce loop as soon as NO path of the whole image is alive
        # (src/pathtracer.cpp:292), which shifts every pixel's stream -- keep the wavefront from running dry
        mb = min(mb, 1)
    opts = dict(spp=int(r.choice([1, 2, 3, 4, 8])), mb=mb, sampler=sampler, edges=int(edges), channels=chans,
                pixel_center=coin(0.15) and not edges, seed=int(r.randint(1, 1000)))
    # with primary edges, anything an edge ray sees must not depend on the filter footprint (the reference reads those
    # rays' differentials at the wrong index, DESIGN.md section 4): constant reflectances and a one-colour sky
    # ... except in a share of the cases, where the vertex / camera gradients are then only compared loosely
    loose = edges and coin(0.3)
    flat = (edges and not loose) or NO_IMAGE_TEXTURES
    # secondary edges: their sample streams are not reproducible, but they only add to vertex gradients -- everything else
    # must still agree exactly
    secondary = mb >= 1 and chans is None and coin(0.25)  # (with extra channels the reference segfaults in its secondary-edge pass)
    opts.update(loose=loose, secondary=secondary)
    env_allowed = not secondary  # (secondary edges next to an environment map crash the reference: stale hit points)
    cam_type = int(r.choice([0, 0, 0, 1, 2, 3]))
    res = (int(r.randint(12, 28)), int(r.randint(12, 28)))
    vp = None
    if coin(0.25) and sampler != "independent":
        y0, x0 = int(r.randint(0, res[0] // 3)), int(r.randint(0, res[1] // 3))
        vp = (y0, x0, int(r.randint(y0 + 4, res[0] + 1)), int(r.randint(x0 + 4, res[1] + 1)))
    cam_grad = coin(0.6)
    pos = [float(r.uniform(-0.6, 0.6)), float(r.uniform(0.8, 1.8)), float(r.uniform(-4.5, -3.2))]
    if cam_type in (2, 3):
        pos = [float(r.uniform(-0.3, 0.3)), float(r.uniform(0.8, 1.4)), float(r.uniform(-1.8, -1.0))]
    look = [float(r.uniform(-0.3, 0.3)), float(r.uniform(0.4, 0.9)), 0.0]
    dist_p = None
    if cam_type == 0 and coin(0.2):
        # (mild lens: with strong coefficients the Gauss-Newton inverse is chaotic near the image corners, in any implementation)
        dist_p = T((r.uniform(-1, 1, 8) * np.array([0.03, 0.005, 0.001, 0.005, 0.001, 0.0003, 0.005, 0.005])).tolist(), cam_grad)
    fov = torch.tensor([float(r.uniform(30, 60))])
    if coin(0.25) and dist_p is None:
        # pose given as a matrix instead of look-at
        p3, l3, u3 = np.array(pos), np.array(look), np.array([0.0, 1.0, 0.0])
        d = (l3 - p3) / np.linalg.norm(l3 - p3)
        rgt = np.cross(u3, d)
        rgt /= np.linalg.norm(rgt)
        nu = np.cross(d, rgt)
        m = np.eye(4)
        m[:3, 0], m[:3, 1], m[:3, 2], m[:3, 3] = rgt, nu, d, p3
        cam = api.Camera(cam_to_world=T(m.tolist(), cam_grad), fov=fov, clip_near=1e-2, resolution=res, viewport=vp, camera_type=cam_type)
    else:
        cam = api.Camera(position=T(pos, cam_grad), look_at=T(look, cam_grad), up=T([0.0, 1.0, 0.0], cam_grad), fov=fov, clip_near=1e-2,
                         resolution=res, viewport=vp, distortion_params=dist_p, camera_type=cam_type)
    cfg.update(cam_type=cam_type, res=res, vp=vp, cam_grad=cam_grad, distort=dist_p is not None, matrix_pose=cam.cam_to_world is not None)

    def texture(ch, lo, hi, size=None, grad=True):
        if coin(0.5) or flat:
            return T(r.uniform(lo, hi, ch).tolist(), grad)
        h, w = size or (int(r.choice([2, 4, 5, 8])), int(r.choice([2, 4, 6, 8])))
        tex = (lo + (hi - lo) * torch.rand(h, w, ch, generator=g)).requires_grad_(grad)
        sc = T(r.uniform(0.5, 3.0, 2).tolist(), coin(0.4))
        return api.Texture(tex, sc)
    shapes, materials, lights = [], [], []
    n_obj = int(r.randint(1, 4))
    for k in range(n_obj):
        spec = coin(0.6)
        nmap = coin(0.25) and not flat
        materials.append(api.Material(diffuse_reflectance=texture(3, 0.1, 0.7), specular_reflectance=texture(3, 0.1, 0.5) if spec else None,
                                      roughness=texture(1, 0.05, 0.6) if spec else None,
                                      normal_map=api.Texture((0.5 + 0.5 * torch.nn.functional.normalize(torch.rand(4, 4, 3, generator=g) * torch.tensor([0.6, 0.6, 0.0]) - torch.tensor([0.3, 0.3, -1.0]), dim=2)).requires_grad_(True)) if nmap else None,
                                      generic_texture=api.Texture(torch.rand(4, 4, int(r.randint(1, 6)), generator=g).requires_grad_(True)) if generic and k == 0 else None,
                                      two_sided=coin(0.4), use_vertex_color=coin(0.15)))
        kind = r.choice(["sphere", "quad", "soup"])
        ctr = (float(r.uniform(-1.0, 1.0)), float(r.uniform(0.4, 1.2)), float(r.uniform(-0.6, 0.8)))
        if kind == "sphere":
            v, i, uv, n = scenes.uv_sphere(dev, float(r.uniform(0.3, 0.6)), ctr, n_theta=int(r.randint(4, 9)), n_phi=int(r.randint(6, 12)), grad=True)
            use_uv, use_n = coin(0.8), coin(0.7)
            cols = torch.rand(v.shape[0], 3, generator=g).requires_grad_(True) if coin(0.5) else None
            uvi = ni = None
            if use_uv and use_n and coin(0.3):  # separate (permuted) uv / normal index buffers
                perm = torch.randperm(uv.shape[0], generator=g)
                inv = torch.empty_like(perm)
                inv[perm] = torch.arange(uv.shape[0])
                uv, n = uv.detach()[perm].requires_grad_(True), n.detach()[perm].requires_grad_(True)
                uvi = inv[i.long()].int().contiguous()
                ni = uvi.clone()
            shapes.append(api.Shape(v, i, k, uvs=uv if use_uv else None, normals=n if use_n else None, colors=cols, uv_indices=uvi, normal_indices=ni))
        elif kind == "quad":
            s = float(r.uniform(0.4, 0.9))
            a = float(r.uniform(0, math.pi))
            ux, uz = math.cos(a) * s, math.sin(a) * s
            v = T([[ctr[0] - ux, ctr[1] - s, ctr[2] - uz], [ctr[0] - ux, ctr[1] + s, ctr[2] - uz], [ctr[0] + ux, ctr[1] - s, ctr[2] + uz], [ctr[0] + ux, ctr[1] + s, ctr[2] + uz]], True)
            uv = T([[0.0, 0.0], [0.0, 1.0], [1.0, 0.0], [1.0, 1.0]], coin(0.5)) if coin(0.7) else None
            shapes.append(api.Shape(v, T([[0, 1, 2], [1, 3, 2]], dt=torch.int32), k, uvs=uv))
        else:
            nt = int(r.randint(3, 12))
            c = (torch.rand(nt, 1, 3, generator=g) - 0.5) * torch.tensor([1.5, 1.0, 1.0]) + torch.tensor(ctr)
            v = (c + 0.5 * (torch.rand(nt, 3, 3, generator=g) - 0.5)).reshape(-1, 3).contiguous().requires_grad_(True)
            shapes.append(api.Shape(v, torch.arange(3 * nt, dtype=torch.int32).reshape(-1, 3).contiguous(), k))
    # floor
    materials.append(api.Material(diffuse_reflectance=texture(3, 0.2, 0.7), two_sided=coin(0.5)))
    shapes.append(api.Shape(T([[-3.0, 0.0, -3.0], [-3.0, 0.0, 3.0], [3.0, 0.0, -3.0], [3.0, 0.0, 3.0]], coin(0.5)), T([[0, 1, 2], [1, 3, 2]], dt=torch.int32), len(materials) - 1,
                            uvs=T([[0.0, 0.0], [0.0, 1.0], [1.0, 0.0], [1.0, 1.0]])))
    materials.append(api.Material(diffuse_reflectance=T([0.0, 0.0, 0.0])))
    env = None
    if coin(0.25) and env_allowed:
        sky = (0.2 + 1.0 * torch.rand(8, 16, 3, generator=g))
        if flat:
            sky = torch.ones(8, 16, 3) * torch.tensor(r.uniform(0.3, 1.0, 3).tolist())
        sky = sky.requires_grad_(True)
        a = float(r.uniform(0, 1))
        e2w = T([[math.cos(a), 0.0, math.sin(a), 0.0], [0.0, 1.0, 0.0, 0.0], [-math.sin(a), 0.0, math.cos(a), 0.0], [0.0, 0.0, 0.0, 1.0]], coin(0.5))
        env = api.EnvironmentMap(sky, e2w, directly_visible=coin(0.8))
    n_l = int(r.randint(0 if env is not None else 1, 3))
    for k in range(n_l):
        c = (float(r.uniform(-1.5, 1.5)), float(r.uniform(2.2, 3.2)), float(r.uniform(-1.0, 1.0)))
        s = float(r.uniform(0.2, 0.7))
        flip = coin(0.3)
        idx = [[0, 1, 2], [1, 3, 2]] if flip else [[0, 2, 1], [1, 2, 3]]
        lamp_mat = len(materials) - 1
        if coin(0.3):  # a lamp that also reflects
            materials.append(api.Material(diffuse_reflectance=T(r.uniform(0.1, 0.6, 3).tolist(), True), two_sided=coin(0.5)))
            lamp_mat = len(materials) - 1
        if coin(0.3):  # a round lamp: many triangles in the area CDF, shading normals on an emitter
            v, i, uv, n = scenes.uv_sphere(dev, s * 0.6, c, n_theta=int(r.randint(3, 6)), n_phi=int(r.randint(4, 8)), grad=coin(0.5))
            shapes.append(api.Shape(v, i, lamp_mat, normals=n if coin(0.5) else None))
            flip = False
        else:
            shapes.append(api.Shape(T([[c[0] - s, c[1], c[2] - s], [c[0] - s, c[1], c[2] + s], [c[0] + s, c[1], c[2] - s], [c[0] + s, c[1], c[2] + s]], coin(0.3)),
                                    T(idx, dt=torch.int32), lamp_mat))
        lights.append(api.AreaLight(len(shapes) - 1, T(r.uniform(5, 25, 3).tolist(), True), two_sided=flip or coin(0.3), directly_visible=coin(0.8)))
    scene = api.Scene(cam, shapes, materials, lights, envmap=env)
    cfg.update(opts, n_obj=n_obj, n_lights=n_l, env=env is not None, generic=generic)
    return scene, cfg


def run(backend, seed):
    from redner_b200 import api
    import parity_utils as pu
    scene, cfg = make_case(seed)
    dev = torch.device("cpu")
    st = backend.SamplerType.sobol if cfg["sampler"] == "sobol" else backend.SamplerType.independent
    chans = [getattr(backend.channels, c) for c in cfg["channels"]] if cfg["channels"] else None
    args = api.RenderFunction.serialize_scene(scene, cfg["spp"], cfg["mb"], channels=chans, sampler_type=st, device=dev, backend=backend,
                                              use_primary_edge_sampling=bool(cfg["edges"]), use_secondary_edge_sampling=bool(cfg["secondary"]),
                                              sample_pixel_center=cfg["pixel_center"])
    img = api.RenderFunction.apply(cfg["seed"], *args)
    grads = {}
    if img.requires_grad:
        w = torch.linspace(0.5, 1.5, img.shape[-1])
        (img * w).pow(2).sum().backward()
        grads = pu.collect_grads(scene)
    return img.detach().numpy(), grads, cfg


STORED_PIXELS = 128


def stored_pixels(img, seed):
    """The pixels of an (H, W, C) image that save_reference keeps: a fixed, seeded sample of STORED_PIXELS of them, as (n, C)."""
    flat = img.reshape(-1, img.shape[-1])
    n = flat.shape[0]
    return flat[np.sort(np.random.RandomState(seed).choice(n, min(n, STORED_PIXELS), replace=False))]


def save_reference(ref, path, first, count):
    """The reference's image (stored_pixels) and gradients of seeds first .. first + count - 1 as float32, packed into one array (one
    zip member per array would double the file): `names` ("<seed>/image", "<seed>/<gradient>"), `shapes` (flattened), `ndims`, `data`."""
    names, arrays = [], []
    for seed in range(first, first + count):
        img, grads, _ = run(ref, seed)
        names.append("%d/image" % seed)
        arrays.append(stored_pixels(img, seed))
        for k, v in grads.items():
            names.append("%d/%s" % (seed, k))
            arrays.append(v.numpy())
    np.savez_compressed(path, names=np.array(names), ndims=np.array([a.ndim for a in arrays], dtype=np.int32),
                        shapes=np.array([d for a in arrays for d in a.shape], dtype=np.int32),
                        data=np.concatenate([a.astype(np.float32).ravel() for a in arrays]))


def stored_reference(path, seed):
    """Image pixels (stored_pixels) and gradients of one seed from a file written by save_reference."""
    z = np.load(path)
    shapes, data = z["shapes"], z["data"]
    pre = "%d/" % seed
    img, grads, dim, off = None, {}, 0, 0
    for name, nd in zip(z["names"], z["ndims"]):
        shape = tuple(int(d) for d in shapes[dim:dim + nd])
        size = int(np.prod(shape))
        if name.startswith(pre):
            a = data[off:off + size].reshape(shape)
            if name == pre + "image":
                img = a
            else:
                grads[name[len(pre):]] = torch.from_numpy(a)
        dim, off = dim + nd, off + size
    return img, grads, make_case(seed)[1]


def main():
    so, first, count = sys.argv[1], int(sys.argv[2]), int(sys.argv[3])
    verbose = "--verbose" in sys.argv
    golden = sys.argv[sys.argv.index("--golden") + 1] if "--golden" in sys.argv else None
    if golden is None:
        import ref_loader
        ref = ref_loader.load()
    from redner_b200 import _lib
    _lib._lib = _lib._bind(ctypes.CDLL(so))
    from redner_b200 import redner as rb
    import parity_utils as pu
    import warnings
    warnings.simplefilter("ignore")
    bad = 0
    for seed in range(first, first + count):
        print("seed", seed, end=" ", flush=True)
        try:
            ir, gr, cfg = stored_reference(golden, seed) if golden else run(ref, seed)
            ic, gc, _ = run(rb, seed)
        except Exception as e:  # noqa: BLE001
            print("ERROR", type(e).__name__, str(e)[:200], flush=True)
            bad += 1
            continue
        e_img = pu.rel_l2(stored_pixels(ic, seed) if golden else ic, ir)
        worst, wk = 0.0, "-"
        missing = set(gr) ^ set(gc)
        scale = max([float(np.linalg.norm(v.numpy())) for v in gr.values()], default=0.0)
        for k in gr:
            if k not in gc:
                continue
            geometric = k.endswith("vertices") or k.startswith("cam.")
            if cfg["edges"] and cfg["sampler"] == "independent" and geometric:
                continue  # PCG edge streams depend on the reference's global compaction order: not reproducible
            if (cfg["loose"] or cfg["secondary"]) and geometric:
                continue
            a, b = gc[k].numpy().astype(np.float64), gr[k].numpy().astype(np.float64)
            # relative to this gradient, but never below the rounding residue of the case's largest gradient
            e = float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-3 * scale, 1e-9))
            if e > worst:
                worst, wk = e, k
        tol = 3e-2 if cfg["edges"] else 1e-3
        flag = e_img > 1e-4 or worst > tol or bool(missing)
        bad += int(flag)
        print("img %.1e grad %.1e (%s)%s" % (e_img, worst, wk, "  <<<<<< " + str(cfg) + (" missing " + str(missing) if missing else "") if flag else ""), flush=True)
        if verbose and not flag:
            print("    ", cfg, flush=True)
    print("flagged", bad, "of", count)


if __name__ == "__main__":
    main()
