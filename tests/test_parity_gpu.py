"""GPU suite: the sm_100a kernels behind the C ABI against the oracle.

 * every golden case (images and gradients produced by the unmodified reference): forward within 1e-4 relative L2
   (north_star tolerance; measured ~2e-7), sample-exact gradients within 1e-3 (measured ~1e-6 .. 1e-4);
 * secondary-edge (shadow) gradients, whose sample streams cannot be reproduced one-to-one: the mean over seeds must agree
   with the reference's mean within the combined standard error;
 * larger configurations and corner features against stored outputs of the reference (pu.GPU_CASES, pu.CORNERS);
 * size-independent properties at the full BASELINE size (512 x 512 x 64 spp): determinism, linearity in the emitted
   radiance, multi-GPU stripes == single image, gradient of a light intensity == image sum identity.
"""
import numpy as np
import pytest
import torch

import parity_utils as pu
import scenes
from redner_b200 import api

pytestmark = pytest.mark.gpu

IMG_TOL = pu.IMG_TOL    # north_star: "within 1e-4 relative L2 at fixed Sobol seed"
GRAD_TOL = pu.GRAD_TOL  # sample-exact gradients (fp32 kernels vs the fp64 reference)


@pytest.fixture(scope="module")
def rb():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from redner_b200 import redner
    return redner


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


@pytest.mark.parametrize("name", list(pu.CASES))
def test_golden_case(rb, dev, name):
    cfg = pu.CASES[name]
    img, grads = pu.render_case(rb, dev, cfg, cfg["seed"])
    pu.assert_matches_golden(name, img.numpy(), grads)


@pytest.mark.parametrize("name", list(pu.GBUFFER_CASES))
def test_gbuffer_golden(rb, dev, name):
    """Forward G-buffer channels (k_forward_channels) against the reference's output, channel by channel; id channels exactly."""
    pu.assert_gbuffer_matches_golden(name, pu.render_gbuffer(rb, dev, pu.GBUFFER_CASES[name]).numpy())


@pytest.mark.parametrize("name", list(pu.SCREEN_CASES))
def test_screen_gradient_golden(rb, dev, name):
    """visualize_screen_gradient: the backward pass with a screen-gradient image attached (first-hit adjoint through the camera
    + primary-edge term), against the reference's output."""
    pu.assert_screen_gradient_matches_golden(name, pu.render_screen_gradient(rb, dev, pu.SCREEN_CASES[name]).numpy())


def test_band_size_does_not_change_gradients(rb, dev, monkeypatch):
    """The adjoint pass walks the image in bands (records through HBM, per-band compaction and sorts): one band or
    hundreds of tiny ones must give the same sample-exact gradients."""
    cfg = dict(pu.CASES["glossy_room_sobol_mb2"], edges=1)
    _, g_one = pu.render_case(rb, dev, cfg, 9)
    monkeypatch.setenv("RB_BAND_BYTES", str(1 << 20))
    _, g_many = pu.render_case(rb, dev, cfg, 9)
    assert set(g_one) == set(g_many)
    for k in g_one:
        assert pu.rel_l2(g_many[k].numpy(), g_one[k].numpy()) < 1e-5, k


def test_lean_and_general_kernels_agree(rb, dev, monkeypatch):
    """Scenes without environment map / special camera / G-buffer run a second, feature-free instantiation of the kernels
    (rb_kernels_lean.cu).  Same source, same samples: image bit-identical, gradients equal up to the order of the atomics."""
    cfg = dict(pu.CASES["glossy_room_sobol_mb2"], edges=1)
    img_lean, g_lean = pu.render_case(rb, dev, cfg, 9)
    monkeypatch.setenv("RB_NO_LEAN", "1")
    img_gen, g_gen = pu.render_case(rb, dev, cfg, 9)
    assert pu.rel_l2(img_lean.numpy(), img_gen.numpy()) < 1e-6
    for k in g_gen:
        assert pu.rel_l2(g_lean[k].numpy(), g_gen[k].numpy()) < 1e-4, k


def test_reference_intersection_known_answer(rb, dev):
    """The reference's own known-answer test for the closest-hit query (test_scene_intersect, src/scene.cpp:761-848): triangle
    (-1,0,1), (1,0,1), (0,1,1); the ray from the origin along +z hits shape 0 / triangle 0 at (0, 0, 1), the ray along -z hits
    nothing.  Driven through the public boundary: a one-pixel pinhole camera at the origin and the G-buffer channels."""
    tri = api.Shape(torch.tensor([[-1.0, 0.0, 1.0], [1.0, 0.0, 1.0], [0.0, 1.0, 1.0]], device=dev), torch.tensor([[0, 1, 2]], dtype=torch.int32, device=dev), 0)
    mat = api.Material(diffuse_reflectance=torch.tensor([0.5, 0.5, 0.5], device=dev))
    chans = [rb.channels.alpha, rb.channels.position, rb.channels.shape_id, rb.channels.triangle_id, rb.channels.depth]
    for look_z, hit in ((1.0, True), (-1.0, False)):
        cam = api.Camera(position=torch.tensor([0.0, 1e-3, 0.0]), look_at=torch.tensor([0.0, 1e-3, look_z]), up=torch.tensor([0.0, 1.0, 0.0]),
                         fov=torch.tensor([1.0]), clip_near=1e-4, resolution=(1, 1))
        sc = api.Scene(cam, [tri], [mat], [])
        args = api.RenderFunction.serialize_scene(sc, 1, 0, channels=chans, device=dev, backend=rb, sample_pixel_center=True)
        px = api.RenderFunction.apply(1, *args).cpu().numpy()[0, 0]
        if hit:
            assert px[0] == 1.0 and np.allclose(px[1:4], [0.0, 1e-3, 1.0], atol=1e-6) and px[4] == 0.0 and px[5] == 0.0 and abs(px[6] - 1.0) < 1e-6
        else:
            assert np.all(px == 0.0)


def test_gbuffer_backward_without_radiance_skips_path_tracing(rb, dev):
    """Deferred set-up (no radiance channel): gradients flow through the first hit and the primary edges only; the
    boundary (secondary-edge) stage and the bounce replay must not run, whatever max_bounces says."""
    sc = scenes.SCENES["single_triangle"](dev, resolution=(24, 24))
    args = api.RenderFunction.serialize_scene(sc, 4, 2, channels=[rb.channels.depth, rb.channels.position], device=dev, backend=rb,
                                              use_secondary_edge_sampling=True)
    img = api.RenderFunction.apply(3, *args)
    img.sum().backward()
    g = pu.collect_grads(sc)
    assert float(g["shape0.vertices"].abs().sum()) > 0 and all(torch.isfinite(v).all() for v in g.values())
    assert float(g["light0.intensity"].abs().sum()) == 0.0


@pytest.mark.parametrize("name", list(pu.STAT_CASES))
def test_secondary_edge_gradients_statistically(rb, dev, name):
    pu.assert_stat_matches_golden(name, pu.render_stat_case(rb, dev, name))


def test_live_reference_if_present(rb, dev):
    """C2 at 128 x 128 x 16 spp without edge sampling: image (fixed pixel sample) and every gradient against the reference's output."""
    name = "c2_shadow_blocker_128_sobol"
    cfg = pu.GPU_CASES[name]
    g = pu.load_golden(name)
    img_c, g_c = pu.render_case(rb, dev, cfg, cfg["seed"])
    img_c = img_c.numpy()
    assert pu.rel_l2(img_c.reshape(-1, img_c.shape[-1])[pu.pixel_sample(img_c.shape)], g["pixels"]) < IMG_TOL
    assert set("grad." + k for k in g_c) == set(k for k in g if k.startswith("grad."))
    for k in g_c:
        assert pu.rel_l2(g_c[k].numpy(), g["grad." + k]) < GRAD_TOL, k


@pytest.mark.parametrize("variant,chans,mb,edges,center", pu.CORNERS)
def test_corner_features_against_live_reference(rb, dev, variant, chans, mb, edges, center):
    """Index buffers for uvs / normals, vertex colours, viewport crops, generic textures, pixel-centre sampling, invisible and
    two-sided lights, deeper paths: image and every gradient against the reference's output."""
    img_c, g_c = pu.render_corner(rb, dev, variant, chans, mb, edges, center)
    g = pu.load_golden("corner_ball_" + variant)
    img_r = g["image"]
    assert img_r.shape == img_c.shape and pu.rel_l2(img_c, img_r) < IMG_TOL
    assert set("grad." + k for k in g_c) == set(k for k in g if k.startswith("grad."))
    for k in g_c:
        r = g["grad." + k]
        if np.linalg.norm(r) > 1e-9:
            assert pu.rel_l2(g_c[k].numpy(), r) < (5e-3 if edges and (k.endswith("vertices") or k.startswith("cam.")) else GRAD_TOL), k


def _render(rb, dev, res, spp, seed=1, intensity_scale=1.0, partition=None, edges=0, scene_fn=scenes.shadow_blocker):
    sc = scene_fn(dev, resolution=(res, res))
    if intensity_scale != 1.0:
        sc.area_lights[0].intensity = (sc.area_lights[0].intensity.detach() * intensity_scale).requires_grad_(True)
    args = api.RenderFunction.serialize_scene(sc, spp, 1, sampler_type=rb.SamplerType.sobol, device=dev, backend=rb,
                                              use_primary_edge_sampling=bool(edges & 1), use_secondary_edge_sampling=bool(edges & 2))
    if partition is None:
        return api.RenderFunction.apply(seed, *args), sc
    c = api.RenderFunction._unpack((seed, seed + 1000003), args)
    c.scene.set_partition(partition[0], partition[1], partition[2])
    img = torch.zeros(res, res, 3, device=dev)
    rb.render(c.scene, c.options, rb.float_ptr(img.data_ptr()), rb.float_ptr(0), None, rb.float_ptr(0), rb.float_ptr(0))
    return img, sc


def test_full_size_properties(rb, dev):
    """BASELINE size (512 x 512 x 64 spp): determinism, linearity, partition union, light-gradient identity."""
    img1, sc = _render(rb, dev, 512, 64)
    img2, _ = _render(rb, dev, 512, 64)
    assert torch.equal(img1, img2), "forward image must be bitwise deterministic (no atomics on the framebuffer)"
    img3, _ = _render(rb, dev, 512, 64, intensity_scale=2.0)
    assert pu.rel_l2(img3.detach().cpu().numpy(), 2 * img1.detach().cpu().numpy()) < 1e-6, "radiance is linear in the light intensity"
    parts = [_render(rb, dev, 512, 64, partition=(p, 4, 16))[0] for p in range(4)]
    union = sum(parts)
    assert torch.equal(union, img1.detach()), "the union of the stripe partitions must equal the single-GPU image bit for bit"
    for p in range(4):
        other = sum(q for i, q in enumerate(parts) if i != p)
        assert float((parts[p] * other).abs().sum()) == 0.0, "stripes must be disjoint"
    # d(sum(img)) / d(intensity_c) * intensity_c == sum(img[..., c])  (the image is linear in the only light's intensity)
    img1.sum().backward()
    gi = sc.area_lights[0].intensity.grad.double()
    lhs = gi * sc.area_lights[0].intensity.detach().double()
    rhs = img1.detach().double().sum((0, 1)).cpu()
    assert torch.allclose(lhs, rhs, rtol=2e-4), (lhs, rhs)


def test_c2_full_size_forward_against_the_reference(rb, dev):
    """The headline configuration itself, C2 at 512 x 512 x 64 spp (forward, fixed Sobol seed): relative L2 within north_star's 1e-4
    against a fixed sample of the reference image's pixels and against its 8 x 8 block means."""
    cfg = pu.GPU_CASES["c2_full_size_forward_pixels"]
    img_c, _ = pu.render_case(rb, dev, cfg, cfg["seed"], backward=False)
    img_c = img_c.numpy()
    blocks = img_c.reshape(64, 8, 64, 8, 3).mean((1, 3))
    g = pu.load_golden("c2_full_size_forward_blocks")["blocks"]
    assert pu.rel_l2(blocks, g) < IMG_TOL, pu.rel_l2(blocks, g)
    px = pu.load_golden("c2_full_size_forward_pixels")["pixels"]
    mine = img_c.reshape(-1, 3)[pu.pixel_sample(img_c.shape)]
    assert pu.rel_l2(mine, px) < IMG_TOL, pu.rel_l2(mine, px)


def _translated_loss(rb, dev, scene, shape, shift, axis, res, spp, seed):
    sc = scenes.SCENES[scene](dev, resolution=(res, res), grad=False)
    v = sc.shapes[shape].vertices.clone()
    v[:, axis] += shift
    sc.shapes[shape].vertices = v
    args = api.RenderFunction.serialize_scene(sc, spp, 1, sampler_type=rb.SamplerType.sobol, device=dev, backend=rb)
    return float(api.RenderFunction.apply(seed, *args).double().sum())


@pytest.mark.parametrize("scene,shape,axes,tol", [("single_triangle", 0, (0, 1), 0.03), ("shadow_blocker", 1, (0,), 0.15)])
def test_gradients_against_finite_differences_end_to_end(rb, dev, scene, shape, axes, tol):
    """End-to-end finite differences (the function-level checks of the reference, src/test_utils.h:15-23 / src/shape.cpp:5-331 /
    src/material.cpp:6-400 / src/camera.cpp:98-475, are restated for our device functions in tests/test_fd_functions_cpu.py).
    Translate a mesh by +-eps: central difference of sum(img) at 256 x 256 x 1024 spp (common random numbers) against the analytic
    gradient sum_v d(sum img)/d(vertex v) with both edge samplers on.
      C1 triangle seen by the camera: interior + primary-edge terms, agree to ~1 %.
      C2 blocker (only its shadow is seen): the secondary-edge term alone.  Along x analytic and finite differences agree within the
      noise; along y / z (towards the lamp) the REFERENCE's estimator itself gives about half of the finite difference
      (profiles/r02_fd_check.txt: reference -471 vs -886, ours -3386 vs -6302 at 256 x 256) -- parity with the reference is pinned
      by the statistical goldens, so only the x axis is asserted here."""
    res, eps, seeds = 256, 0.02, (1, 2, 3, 4)
    analytic = np.zeros(3)
    for seed in seeds:
        sc = scenes.SCENES[scene](dev, resolution=(res, res))
        args = api.RenderFunction.serialize_scene(sc, 256, 1, sampler_type=rb.SamplerType.sobol, device=dev, backend=rb)
        api.RenderFunction.apply(seed, *args).sum().backward()
        analytic += sc.shapes[shape].vertices.grad.double().sum(0).cpu().numpy() / len(seeds)
    for axis in axes:
        fd = np.mean([(_translated_loss(rb, dev, scene, shape, eps, axis, res, 1024, s) - _translated_loss(rb, dev, scene, shape, -eps, axis, res, 1024, s)) / (2 * eps)
                      for s in seeds])
        assert abs(analytic[axis] - fd) < tol * max(abs(fd), 0.1 * np.abs(analytic).max()), (axis, analytic, fd)


def test_ragged_and_degenerate_inputs(rb, dev):
    # spp that is not a power of two, non-square viewport crop, max_bounces 0, a scene without lights
    sc = scenes.shadow_blocker(dev, resolution=(37, 53))
    sc.camera.viewport = (3, 5, 31, 47)
    args = api.RenderFunction.serialize_scene(sc, 5, 1, sampler_type=rb.SamplerType.sobol, device=dev, backend=rb)
    img = api.RenderFunction.apply(1, *args)
    assert tuple(img.shape) == (28, 42, 3) and torch.isfinite(img).all() and float(img.sum()) > 0
    img.sum().backward()
    args0 = api.RenderFunction.serialize_scene(scenes.shadow_blocker(dev, resolution=(16, 16)), 3, 0, device=dev, backend=rb)
    img0 = api.RenderFunction.apply(1, *args0)
    assert float(img0.abs().sum()) == 0.0  # the light is outside the view; without bounces nothing is lit
    dark = scenes.shadow_blocker(dev, resolution=(16, 16))
    dark.area_lights = []
    for s in dark.shapes:
        s.light_id = -1
    imgd = api.RenderFunction.apply(1, *api.RenderFunction.serialize_scene(dark, 2, 2, device=dev, backend=rb))
    assert float(imgd.abs().sum()) == 0.0
    with pytest.raises(RuntimeError):
        api.RenderFunction.apply(1, *api.RenderFunction.serialize_scene(scenes.single_triangle(dev, resolution=(8, 8)), 1, 1, device=dev, backend=rb,
                                                                         channels=[rb.channels.radiance, rb.channels.radiance]))


def test_bvh_stress_against_live_reference(rb, dev):
    cfg = pu.GPU_CASES["bvh_stress_random_soup"]
    img_c, _ = pu.render_case(rb, dev, cfg, cfg["seed"], backward=False)
    img_c = img_c.numpy()
    g = pu.load_golden("bvh_stress_random_soup")
    px_c, px_r = img_c.reshape(-1, 3)[pu.pixel_sample(img_c.shape)], g["pixels"]
    # 2000 intersecting random triangles: a handful of silhouette samples may resolve differently in fp32
    assert pu.rel_l2(px_c, px_r) < 5e-3
    d = np.abs(px_c - px_r).max(-1)
    assert (d > 1e-3 * g["image_max"]).mean() < 2e-3
