"""Shared helpers of the parity tests and the golden generator: the list of golden cases and one function that
renders a case (image + gradients of loss = sum(img^2)) with ANY module exposing the `redner` surface."""
import os

import numpy as np
import torch

import scenes
from redner_b200 import api

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

# edges: bit 0 primary edge sampling, bit 1 secondary edge sampling
CASES = {
    # C1 geometry (tests/test_single_triangle.py), primary-edge gradients are sample-exact
    "c1_single_triangle_sobol": dict(scene="single_triangle", res=64, spp=4, mb=1, sampler="sobol", edges=1, seed=1),
    "c1_single_triangle_pcg": dict(scene="single_triangle", res=48, spp=4, mb=1, sampler="independent", edges=0, seed=3),
    # C2 geometry (tests/test_shadow_blocker.py) without edge sampling: every gradient is sample-exact
    "c2_shadow_blocker_sobol": dict(scene="shadow_blocker", res=96, spp=16, mb=1, sampler="sobol", edges=0, seed=2),
    # glossy textured room: specular lobe, shading normals, uvs, mip-mapped textures, two lights, 2 bounces
    "glossy_room_sobol_mb2": dict(scene="glossy_room", res=48, spp=8, mb=2, sampler="sobol", edges=0, seed=5),
    "glossy_room_pcg_mb3": dict(scene="glossy_room", res=32, spp=4, mb=3, sampler="independent", edges=0, seed=7),
    # primary edges on a smooth, uv-seamed mesh behind / in front of other geometry: hidden-edge rejection (an edge sample
    # counts only if one of its two rays sees a face of the edge) and the order of duplicated seam edges.  Rays graze the
    # silhouette by construction, so a few hit decisions differ between any two BVHs -- the reference itself changes by
    # ~1e-4 between two runs (Embree's parallel build) -- hence the looser tolerance on the vertex gradient.
    "glossy_room_primary_edges": dict(scene="glossy_room", res=40, spp=8, mb=1, sampler="sobol", edges=1, seed=13, vertex_tol=5e-3),
    # adjoints of the G-buffer channels (deferred rendering), interior + primary edges: src/primary_contribution.cpp:438-713,
    # channel multipliers of the edge integrand src/edge.cpp:476-481
    "gbuffer_bwd_glossy_room": dict(scene="glossy_room", res=32, spp=4, mb=1, sampler="sobol", edges=1, seed=4, vertex_tol=5e-3,
                                    channels=["radiance", "alpha", "depth", "position", "geometry_normal", "shading_normal", "uv", "barycentric_coordinates",
                                              "diffuse_reflectance", "specular_reflectance", "roughness", "shape_id"]),
    # no radiance channel at all, max_bounces 0 (the deferred-shading set-up of the tutorials); camera gradients included
    "gbuffer_bwd_single_triangle_no_radiance": dict(scene="single_triangle", res=32, spp=4, mb=0, sampler="sobol", edges=1, seed=7,
                                                    channels=["depth", "alpha", "position", "uv"]),
    # environment map: importance-sampled light + BSDF-miss lookups with MIS, sky seen directly by the camera, gradients of
    # the map's texels and of its rotation (src/envmap.h, src/path_contribution.cpp:51-118,295-337,520-590)
    "env_ball_sobol_mb2": dict(scene="env_ball", res=40, spp=8, mb=2, sampler="sobol", edges=0, seed=21),
    # the sky seen directly through a fisheye lens with a differentiable pose: of a primary ray that leaves the scene only the
    # direction adjoint reaches the camera, the footprint adjoint does not (src/primary_intersection.cpp:9-16,:30-41); low
    # resolution so that the sky is filtered from coarse mip levels and the footprint matters
    "env_ball_fisheye_camera": dict(scene="env_ball_fisheye", res=16, spp=4, mb=0, sampler="sobol", edges=0, seed=23),
    # primary edges against the sky.  Sample-exact only for a sky without mip dependence: the reference looks edge rays'
    # differentials up at the wrong index (written at [idx], read at [2 idx + side]: src/edge.cpp:443-444 vs :608), so the
    # filter footprint of anything an edge ray sees is stale data there; we use the differential of the edge point.
    "env_ball_flat_sky_primary_edges": dict(scene="env_ball_flat_sky", res=40, spp=8, mb=1, sampler="sobol", edges=1, seed=22, vertex_tol=5e-3),
    # fisheye (equi-angular) and panorama cameras from inside the room, differentiable pose, primary edges sampled on the
    # camera-space film (src/camera.h:154-197,343-498,533-553,669-724; src/edge.cpp:486-592,737-757)
    "fisheye_room_primary_edges": dict(scene="fisheye_room", res=40, spp=4, mb=1, sampler="sobol", edges=1, seed=31, vertex_tol=5e-3),
    "panorama_room_primary_edges": dict(scene="panorama_room", res=40, spp=4, mb=1, sampler="sobol", edges=1, seed=32, vertex_tol=5e-3),
    # Brown-Conrady lens distortion (src/camera_distortion.h): rays through inverse_distort (Gauss-Newton), projection
    # through distort, parameter gradients by the implicit function theorem, primary edges on the non-linear path
    "distort_room_primary_edges": dict(scene="distort_room", res=40, spp=4, mb=1, sampler="sobol", edges=1, seed=34, vertex_tol=5e-3, cam_tol=5e-3),
    # orthographic camera: all primary-edge rays are parallel and graze the silhouettes, the pose gradient is the sum of those
    # few samples -- the reference itself moves by up to 1e-3 between two runs on it (Embree's parallel BVH build)
    "ortho_room_primary_edges": dict(scene="ortho_room", res=40, spp=4, mb=1, sampler="sobol", edges=1, seed=33, vertex_tol=5e-3, cam_tol=2e-2),
    # ---- BASELINE configs C3 / C4 on the reference's own meshes (fixtures exported by tests/golden/export_ref_scenes.py), reduced size
    # C3 tests/test_teapot_reflectance.py: 15 712 triangles, textured floor, 3 lamps, glossy teapot; SVBRDF + camera-pose gradients
    "c3_teapot_sobol_mb2": dict(scene="teapot", res=64, spp=4, mb=2, sampler="sobol", edges=0, seed=3),
    # ... with primary edges (the pose gradient is dominated by them; grazing edge rays: see glossy_room_primary_edges)
    "c3_teapot_primary_edges": dict(scene="teapot", res=96, spp=4, mb=2, sampler="sobol", edges=1, seed=5, cam_tol=1e-2),
    # C4 tests/test_bunny_box.py: closed Cornell-style box, 14 416 triangles, max_bounces 5, bunny vertices differentiable.  pyredner's
    # default sampler (independent) with the file's camera; Sobol with the camera moved off the box's axis (scenes.bunny_box_shifted:
    # on the axis Sobol points put primary rays exactly on edges shared by two shapes, a tie decided by the last bit in any tracer)
    "c4_bunny_box_pcg_mb5": dict(scene="bunny_box", res=48, spp=4, mb=5, sampler="independent", edges=0, seed=4),
    "c4_bunny_box_shifted_sobol_mb5": dict(scene="bunny_box_shifted", res=48, spp=4, mb=5, sampler="sobol", edges=0, seed=4),
    # primary edges on the bunny's silhouette: ~13 of 32 k edge samples resolve their grazing rays differently from Embree (one
    # vertex each), measured 0.7 - 1.3e-2 on the vertex gradient; the reference is bit-stable between runs on this scene
    "c4_bunny_box_shifted_primary_edges": dict(scene="bunny_box_shifted", res=64, spp=8, mb=5, sampler="sobol", edges=1, seed=9, vertex_tol=3e-2),
    # normal-mapped ball with a mip-mapped specular texture and a differentiable uv_scale
    "nmap_room_sobol_mb2": dict(scene="nmap_room", res=40, spp=8, mb=2, sampler="sobol", edges=0, seed=11),
}
# forward-only G-buffer renders (src/channels.cpp, src/pathtracer.cpp:44-175); channel names of the `redner.channels` enum.
# The second case puts radiance LAST to pin the reference's "channel index used as float offset" behaviour.
GBUFFER_CASES = {
    "gbuffer_glossy_room": dict(scene="glossy_room", res=40, spp=4, mb=1, sampler="sobol", seed=4,
                                channels=["radiance", "alpha", "depth", "position", "geometry_normal", "shading_normal", "uv", "barycentric_coordinates",
                                          "diffuse_reflectance", "specular_reflectance", "roughness", "shape_id", "triangle_id", "material_id"]),
    "gbuffer_nmap_room_radiance_last": dict(scene="nmap_room", res=32, spp=4, mb=1, sampler="sobol", seed=6,
                                            channels=["depth", "shading_normal", "radiance"]),
}
# d(image) / d(screen position of each pixel) (RenderFunction.visualize_screen_gradient): first-hit adjoint through the camera
# plus the primary-edge term (src/primary_intersection.cpp:104-114, src/edge.cpp:765-773)
SCREEN_CASES = {
    "screen_gradient_c1": dict(scene="single_triangle", res=32, spp=4, mb=1, sampler="sobol", edges=1, seed=5, tol=1e-4),
    # (textured floor seen by edge rays: the stale-footprint difference of the primary-edge entries above applies)
    "screen_gradient_fisheye_room": dict(scene="fisheye_room", res=24, spp=2, mb=1, sampler="sobol", edges=1, seed=5, tol=3e-3),
}
# Secondary-edge gradients SAMPLE BY SAMPLE: only the host build of the device headers with -DRB_EMU_REF_STREAMS can index the
# boundary-sample streams by the rank of the pixel in the reference's compacted wavefront (src/pathtracer.cpp:504-505); with
# that, every gradient of these cases equals the reference's (measured 1e-7 .. 4e-6).  Not run on the GPU.
REFSTREAM_CASES = {
    "c1_secondary_exact": dict(scene="single_triangle", res=32, spp=4, mb=2, sampler="sobol", edges=2, seed=2),
    "c2_all_vertices_secondary_exact": dict(scene="shadow_blocker_all", res=32, spp=8, mb=2, sampler="sobol", edges=2, seed=1),
    "c1_both_edge_samplers_exact": dict(scene="single_triangle", res=32, spp=4, mb=1, sampler="sobol", edges=3, seed=2),
}
STAT_CASES = {
    # secondary-edge (shadow) gradient of the blocker: mean over seeds +- standard error
    "c2_shadow_blocker_secondary_stat": dict(scene="shadow_blocker", res=64, spp=64, mb=1, sampler="sobol", edges=3, seeds=list(range(1, 9)),
                                             keys=["shape1.vertices"]),
    # every vertex of C2 differentiable, FEW samples per pixel, many seeds: the mean over seeds at a fixed low sample count
    # depends on how the reference consumes its (jointly scrambled, hence related) Sobol dimensions, in particular on its
    # per-sample strategy coin (src/edge.cpp:1461-1472); compared component by component (`z_rms`)
    "c2_all_vertices_secondary_stat": dict(scene="shadow_blocker_all", res=32, spp=8, mb=1, sampler="sobol", edges=2, seeds=list(range(1, 65)),
                                           keys=["shape0.vertices", "shape1.vertices", "shape2.vertices"], z_rms=2.0),
    # boundary terms on the reference's meshes: teapot (lid + body vertices, 3 lamps, 2 bounces) and the bunny in its box
    # (compared on the gradient w.r.t. a rigid motion of each shape, `reduce="rigid"`)
    "c3_teapot_secondary_stat": dict(scene="teapot_geometry", res=48, spp=8, mb=2, sampler="sobol", edges=2, seeds=list(range(1, 49)),
                                     keys=["shape4.vertices", "shape5.vertices"], reduce="rigid", test="ranks"),
    "c4_bunny_box_secondary_stat": dict(scene="bunny_box_shifted", res=48, spp=8, mb=2, sampler="sobol", edges=2, seeds=list(range(1, 49)),
                                        keys=["shape6.vertices"], reduce="rigid", test="ranks"),
    "glossy_room_secondary_stat": dict(scene="glossy_room", res=32, spp=32, mb=2, sampler="sobol", edges=3, seeds=list(range(1, 25)),
                                       keys=["shape3.vertices"]),
}


def _res(cfg):
    """`res` is the side of a square image or an explicit (height, width)."""
    r = cfg["res"]
    return tuple(r) if isinstance(r, (tuple, list)) else (r, r)


def collect_grads(scene):
    out = {}
    cam = scene.camera
    for k in ("position", "look_at", "up", "distortion_params"):
        t = getattr(cam, k)
        if t is not None and t.grad is not None:
            out["cam." + k] = t.grad.detach().cpu().clone()
    for i, s in enumerate(scene.shapes):
        for k in ("vertices", "uvs", "normals", "colors"):
            t = getattr(s, k)
            if t is not None and t.grad is not None:
                out["shape%d.%s" % (i, k)] = t.grad.detach().cpu().clone()
    for i, m in enumerate(scene.materials):
        for k in ("diffuse_reflectance", "specular_reflectance", "roughness", "normal_map", "generic_texture"):
            t = getattr(m, k)
            if t is not None and t.texels.grad is not None:
                out["mat%d.%s" % (i, k)] = t.texels.grad.detach().cpu().clone()
            if t is not None and t.uv_scale.grad is not None:
                out["mat%d.%s.uv_scale" % (i, k)] = t.uv_scale.grad.detach().cpu().clone()
    env = getattr(scene, "envmap", None)
    if env is not None:
        if env.values.texels.grad is not None:
            out["envmap.values"] = env.values.texels.grad.detach().cpu().clone()
        if env.env_to_world.grad is not None:
            out["envmap.env_to_world"] = env.env_to_world.grad.detach().cpu().clone()
    for i, l in enumerate(scene.area_lights):
        if l.intensity.grad is not None:
            out["light%d.intensity" % i] = l.intensity.grad.detach().cpu().clone()
    return out


def render_case(backend, device, cfg, seed, backward=True):
    sc = scenes.SCENES[cfg["scene"]](device, resolution=_res(cfg))
    st = backend.SamplerType.sobol if cfg["sampler"] == "sobol" else backend.SamplerType.independent
    chans = [getattr(backend.channels, c) for c in cfg["channels"]] if "channels" in cfg else None
    args = api.RenderFunction.serialize_scene(sc, cfg["spp"], cfg["mb"], channels=chans, sampler_type=st, device=device, backend=backend,
                                              use_primary_edge_sampling=bool(cfg["edges"] & 1),
                                              use_secondary_edge_sampling=bool(cfg["edges"] & 2))
    img = api.RenderFunction.apply(seed, *args)
    grads = {}
    if backward and img.requires_grad:
        # G-buffer cases weight the image dimensions differently so that no channel's adjoint can hide behind another's
        w = torch.linspace(0.5, 1.5, img.shape[-1], device=img.device) if chans is not None else 1.0
        (img * w).pow(2).sum().backward()
        grads = collect_grads(sc)
    return img.detach().cpu(), grads


def render_gbuffer(backend, device, cfg):
    sc = scenes.SCENES[cfg["scene"]](device, resolution=_res(cfg), grad=False)
    st = backend.SamplerType.sobol if cfg["sampler"] == "sobol" else backend.SamplerType.independent
    chans = [getattr(backend.channels, c) for c in cfg["channels"]]
    args = api.RenderFunction.serialize_scene(sc, cfg["spp"], cfg["mb"], channels=chans, sampler_type=st, device=device, backend=backend)
    return api.RenderFunction.apply(cfg["seed"], *args).detach().cpu()


def rel_l2(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    n = np.linalg.norm(b)
    return float(np.linalg.norm(a - b) / n) if n > 0 else float(np.linalg.norm(a - b))


def load_golden(name):
    return dict(np.load(os.path.join(GOLDEN_DIR, name + ".npz")))


IMG_TOL = 1e-4   # north_star: "within 1e-4 relative L2 at fixed Sobol seed"
GRAD_TOL = 1e-3  # sample-exact gradients (fp32 kernels vs the fp64 reference)
CHANNEL_WIDTH = {"radiance": 3, "alpha": 1, "depth": 1, "position": 3, "geometry_normal": 3, "shading_normal": 3, "uv": 2, "barycentric_coordinates": 2,
                 "diffuse_reflectance": 3, "specular_reflectance": 3, "roughness": 1, "shape_id": 1, "triangle_id": 1, "material_id": 1}


def assert_matches_golden(name, img, grads):
    """Image and every gradient of golden case `name` (numpy image, dict of torch gradients) within the suite's tolerances."""
    cfg = CASES[name] if name in CASES else REFSTREAM_CASES[name]
    g = load_golden(name)
    assert rel_l2(img, g["image"]) < IMG_TOL
    exact_vertices = not (cfg["sampler"] == "independent" and cfg["edges"])  # PCG edge streams depend on global compaction
    assert set("grad." + k for k in grads) == set(k for k in g if k.startswith("grad.")), name
    for k, v in grads.items():
        ref = g["grad." + k]
        if np.linalg.norm(ref) < 1e-9:  # a gradient that is exactly zero up to rounding (e.g. rotating a one-colour sky)
            assert np.linalg.norm(v.numpy()) < 1e-4, k
        elif k.endswith("vertices") and not exact_vertices:
            assert rel_l2(v.numpy(), ref) < 0.5, k
        elif k.startswith("cam.") and "cam_tol" in cfg:
            assert rel_l2(v.numpy(), ref) < cfg["cam_tol"], (k, rel_l2(v.numpy(), ref))
        elif k.endswith("vertices") and "vertex_tol" in cfg:
            assert rel_l2(v.numpy(), ref) < cfg["vertex_tol"], (k, rel_l2(v.numpy(), ref))
        else:
            assert rel_l2(v.numpy(), ref) < GRAD_TOL, (k, rel_l2(v.numpy(), ref))


def assert_gbuffer_matches_golden(name, img):
    """Forward G-buffer channels against the reference's output, channel by channel; id channels exactly."""
    cfg = GBUFFER_CASES[name]
    g = load_golden(name)["image"]
    assert img.shape == g.shape
    assert rel_l2(img, g) < IMG_TOL
    if cfg["channels"][0] == "radiance":  # otherwise radiance overlaps other channels (reference quirk, reproduced: whole-image check above)
        d = 0
        for c in cfg["channels"]:
            n = CHANNEL_WIDTH[c]
            if c.endswith("_id"):
                assert np.array_equal(img[..., d:d + n], g[..., d:d + n]), c
            else:
                assert rel_l2(img[..., d:d + n], g[..., d:d + n]) < IMG_TOL, c
            d += n


def assert_stat_matches_golden(name, acc):
    """Mean over seeds of the gradients in `acc` ({key: [array per seed]}) against the reference's mean +- standard error."""
    cfg = STAT_CASES[name]
    g = load_golden(name)
    for k in cfg["keys"]:
        a = np.stack(acc[k]).astype(np.float64)
        if cfg.get("test") == "ranks":
            # Boundary terms on real meshes are heavy-tailed (single samples with tiny pdfs dominate the mean of a run), so the mean
            # over seeds is no usable statistic.  Two-sample rank test per component instead: the per-seed values of the two
            # implementations must come from the same distribution (Mann-Whitney U, no component below p = 1e-3, median p not small),
            # and the medians must agree within 4 robust standard errors.
            from scipy.stats import mannwhitneyu
            r = g["samples." + k].astype(np.float64)
            ps = np.array([mannwhitneyu(a[:, i], r[:, i], alternative="two-sided").pvalue for i in range(a.shape[1])])
            assert ps.min() > 1e-3 and np.median(ps) > 0.05, (k, ps)
            se = lambda x: 1.2533 * 1.4826 * np.median(np.abs(x - np.median(x, 0)), 0) / np.sqrt(x.shape[0])
            zmed = (np.median(a, 0) - np.median(r, 0)) / np.sqrt(se(a) ** 2 + se(r) ** 2)
            assert np.abs(zmed).max() < 4.0, (k, zmed)
            continue
        mean, sem = a.mean(0), a.std(0, ddof=1) / np.sqrt(a.shape[0])
        ref_mean, ref_sem = g["mean." + k], g["sem." + k]
        err = np.linalg.norm(mean - ref_mean)
        noise = np.sqrt(np.linalg.norm(sem) ** 2 + np.linalg.norm(ref_sem) ** 2)
        assert err < 4 * noise, (k, err, noise)
        assert err < 0.35 * np.linalg.norm(ref_mean), (k, err, np.linalg.norm(ref_mean))
        if "z_rms" in cfg:  # per component; the floor keeps exactly-zero components (rounding residue) out of it
            floor = 1e-3 * np.abs(ref_mean).max()
            z = (mean - ref_mean) / np.maximum(np.sqrt(sem ** 2 + ref_sem ** 2), floor)
            assert np.sqrt((z ** 2).mean()) < cfg["z_rms"], (k, float(np.sqrt((z ** 2).mean())), float(np.abs(z).max()))
            assert np.abs(z).max() < 5.0, (k, float(np.abs(z).max()))


def _rigid_reduce(cfg, key, g):
    """Gradient of a vertex buffer -> gradient w.r.t. a rigid motion of the whole shape: translation sum(g) and rotation about the
    centroid sum((v - c) x g) -- the parameters tests/test_bunny_box.py optimises; far less noisy than 3 x 7 000 components."""
    sc = scenes.SCENES[cfg["scene"]](torch.device("cpu"), resolution=_res(cfg), grad=False)
    v = sc.shapes[int(key.split(".")[0][5:])].vertices.detach().cpu().numpy().astype(np.float64)
    g = g.astype(np.float64)
    return np.concatenate([g.sum(0), np.cross(v - v.mean(0), g).sum(0)])


def render_stat_case(backend, device, name):
    cfg = STAT_CASES[name]
    acc = {k: [] for k in cfg["keys"]}
    for seed in cfg["seeds"]:
        _, grads = render_case(backend, device, cfg, seed)
        for k in cfg["keys"]:
            g = grads[k].numpy()
            acc[k].append(_rigid_reduce(cfg, k, g) if cfg.get("reduce") == "rigid" else g)
    return acc


def render_screen_gradient(backend, device, cfg):
    sc = scenes.SCENES[cfg["scene"]](device, resolution=_res(cfg), grad=False)
    st = backend.SamplerType.sobol if cfg["sampler"] == "sobol" else backend.SamplerType.independent
    return api.visualize_screen_gradient(None, cfg["seed"], sc, cfg["spp"], cfg["mb"], sampler_type=st, use_primary_edge_sampling=bool(cfg["edges"] & 1),
                                         use_secondary_edge_sampling=bool(cfg["edges"] & 2), device=device, backend=backend).detach().cpu()


def assert_screen_gradient_matches_golden(name, img):
    g = load_golden(name)["image"]
    assert img.shape == g.shape and np.linalg.norm(g) > 0
    assert rel_l2(img, g) < SCREEN_CASES[name]["tol"], rel_l2(img, g)


# Larger configurations that only the GPU suite renders (tests/test_parity_gpu.py); the reference's outputs are stored under
# the key's name.  Images larger than a few thousand pixels are stored as a fixed, seeded sample of PIXEL_SAMPLE pixels.
GPU_CASES = {
    "c2_shadow_blocker_128_sobol": dict(scene="shadow_blocker", res=128, spp=16, mb=1, sampler="sobol", edges=0, seed=11),
    # 2000 intersecting random triangles (forward only)
    "bvh_stress_random_soup": dict(scene="random_soup", res=128, spp=4, mb=2, sampler="sobol", edges=0, seed=4),
    # the headline configuration itself, C2 at 512 x 512 x 64 spp (forward only)
    "c2_full_size_forward_pixels": dict(scene="shadow_blocker", res=512, spp=64, mb=1, sampler="sobol", edges=0, seed=1),
}
PIXEL_SAMPLE = 4096


def pixel_sample(shape, seed=0):
    """Flat indices of the fixed pixel sample of an (H, W, C) image."""
    return np.sort(np.random.RandomState(seed).choice(shape[0] * shape[1], PIXEL_SAMPLE, replace=False))


def envmap_table_inputs():
    """The seeded sky and rotation whose environment-map tables are stored as pyredner_envmap_tables.npz."""
    g = torch.Generator().manual_seed(3)
    sky = 0.1 + 2.0 * torch.rand(12, 24, 3, generator=g)
    e2w = torch.tensor([[0.8, 0.0, 0.6, 0.0], [0.0, 1.0, 0.0, 0.0], [-0.6, 0.0, 0.8, 0.0], [0.0, 0.0, 0.0, 1.0]])
    return sky, e2w


CORNERS = [  # (variant, channels, max_bounces, primary edges, sample_pixel_center)
    ("vcolor", ["radiance", "vertex_color", "diffuse_reflectance"], 1, True, False),
    ("viewport", ["radiance"], 2, True, False),
    ("plain", ["radiance", "uv", "shading_normal"], 1, False, True),
    ("generic", ["radiance", "generic_texture"], 1, False, False),  # (the reference corrupts its heap with generic textures + edges)
    ("invisible", ["radiance"], 3, True, False),
]


def render_corner(backend, device, variant, chans, mb, edges, center):
    """scenes.corner_ball: image and every gradient of sum((img * w)^2), w weighting the channels differently."""
    sc = scenes.corner_ball(device, variant=variant)
    ch = [getattr(backend.channels, c) for c in chans]
    args = api.RenderFunction.serialize_scene(sc, 4, mb, channels=ch, sampler_type=backend.SamplerType.sobol, device=device, backend=backend,
                                              use_primary_edge_sampling=edges, use_secondary_edge_sampling=False, sample_pixel_center=center)
    img = api.RenderFunction.apply(3, *args)
    w = torch.linspace(0.5, 1.5, img.shape[-1], device=img.device)
    (img * w).pow(2).sum().backward()
    return img.detach().cpu().numpy(), collect_grads(sc)
