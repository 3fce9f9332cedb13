"""CPU suite, part 3: host-side logic.

 * the host mirror of the pyredner interface (redner_b200/api.py) drives a `redner` module correctly -- the UNMODIFIED reference
   module where oracle/_ref is built, and the shim on the host build of the device headers: argument marshalling,
   gradient-tuple alignment (one entry per serialized argument), seeds;
 * the `redner` shim marshals descriptors the way the reference's constructors read them;
 * the multi-GPU host logic (stripe partition, packed all-reduce, data-parallel pose loop) with the gloo backend and
   world_size 2.
"""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import parity_utils as pu
import scenes
from redner_b200 import api
from redner_b200 import dist as rdist


@pytest.fixture
def emu_backend(monkeypatch):
    """The `redner` shim bound, for one test, to the host build of the device headers (tools/cpu_emu, test infrastructure)."""
    import ctypes
    import test_device_code_cpu as tdc
    from redner_b200 import _lib, redner as rb
    monkeypatch.setattr(_lib, "_lib", _lib._bind(ctypes.CDLL(tdc._build())))
    return rb


def _check_one_gradient_per_argument(backend):
    sc = scenes.glossy_room(torch.device("cpu"), resolution=(8, 8))
    args = api.RenderFunction.serialize_scene(sc, 1, 1, device=torch.device("cpu"), backend=backend)
    img = api.RenderFunction.apply(3, *args)
    img.sum().backward()  # autograd itself checks len(grads) == len(inputs)
    assert sc.shapes[3].vertices.grad is not None and sc.area_lights[0].intensity.grad is not None
    assert sc.materials[0].diffuse_reflectance.texels.grad.shape == sc.materials[0].diffuse_reflectance.texels.shape


def _check_seed_convention(backend):
    """backward seed = forward seed + 1000003 unless correlated random numbers are requested
    (pyredner/render_pytorch.py:658-663)."""
    sc = scenes.single_triangle(torch.device("cpu"), resolution=(8, 8))
    args = api.RenderFunction.serialize_scene(sc, 1, 1, device=torch.device("cpu"), backend=backend)
    c = api.RenderFunction._unpack((5, 5 + 1000003), args)
    assert c.seed == (5, 1000008) and c.options.seed == 5


def test_backward_returns_one_gradient_per_argument(emu_backend):
    _check_one_gradient_per_argument(emu_backend)


def test_backward_returns_one_gradient_per_argument_on_the_reference_module(reference_module):
    _check_one_gradient_per_argument(reference_module)


def test_seed_convention(emu_backend):
    _check_seed_convention(emu_backend)


def test_seed_convention_on_the_reference_module(reference_module):
    _check_seed_convention(reference_module)


def test_shim_marshalling_matches_reference_constructor_order():
    from redner_b200 import redner as rb
    pos = torch.tensor([1.0, 2.0, 3.0])
    look = torch.tensor([0.0, 0.5, 0.0])
    up = torch.tensor([0.0, 1.0, 0.0])
    k = torch.eye(3).contiguous()
    cam = rb.Camera(64, 32, rb.float_ptr(pos.data_ptr()), rb.float_ptr(look.data_ptr()), rb.float_ptr(up.data_ptr()), rb.float_ptr(0), rb.float_ptr(0),
                    rb.float_ptr(k.data_ptr()), rb.float_ptr(k.data_ptr()), rb.float_ptr(0), 1e-2, rb.CameraType.perspective, rb.Vector2i(0, 0),
                    rb.Vector2i(64, 32))
    assert cam.use_look_at and not cam.has_distortion_params()
    assert list(cam._c.position) == [1.0, 2.0, 3.0] and (cam._c.width, cam._c.height) == (64, 32)
    assert list(cam._c.viewport_end) == [64, 32]
    inten = torch.tensor([1.0, 2.0, 3.0])
    al = rb.AreaLight(2, rb.float_ptr(inten.data_ptr()), True, False)
    assert list(al._c.intensity) == [1.0, 2.0, 3.0] and al._c.two_sided == 1 and al._c.directly_visible == 0
    t = rb.Texture3([rb.float_ptr(16)], [0], [0], 3, rb.float_ptr(32))
    assert t._c.num_levels == 1 and t._c.width[0] == 0 and t._c.channels == 3
    m = rb.Material(t, t, rb.Texture1([rb.float_ptr(16)], [0], [0], 1, rb.float_ptr(32)), rb.TextureN([], [], [], 0, rb.float_ptr(0)),
                    rb.Texture3([], [], [], 3, rb.float_ptr(0)), True, False, False)
    assert m.get_diffuse_levels() == 1 and m.get_normal_map_levels() == 0 and m.get_diffuse_size(0) == (0, 0)


def test_stripe_partition_covers_every_row_once():
    for h, world, rps in ((512, 8, 16), (100, 3, 7), (5, 4, 2), (64, 1, 16)):
        seen = []
        for r in range(world):
            seen += rdist.owned_rows(h, r, world, rps)
        assert sorted(seen) == list(range(h))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        # (1) packed all-reduce == per-tensor sums
        a, b = torch.full((3, 2), float(rank + 1)), torch.arange(5, dtype=torch.float32) * (rank + 1)
        ra, rb_ = rdist.all_reduce_packed([a, b])
        tot = sum(range(1, world + 1))
        ok = torch.equal(ra, torch.full((3, 2), float(tot))) and torch.equal(rb_, torch.arange(5, dtype=torch.float32) * tot)
        # (2) tile sharding: every rank fills only its stripes; the all-reduced framebuffer is the full image
        h, w = 37, 5
        full = torch.arange(h * w, dtype=torch.float32).reshape(h, w, 1)
        mine = torch.zeros_like(full)
        rows = rdist.owned_rows(h, rank, world, 4)
        mine[rows] = full[rows]
        dist.all_reduce(mine)
        ok = ok and torch.equal(mine, full)
        # (3) data-parallel pose loop: gradients of sum_p (x * (p + 1))^2 w.r.t. x, poses split across ranks
        x = torch.tensor([2.0, -1.0], requires_grad=True)
        n_poses = 5
        _, (gx,) = rdist.render_poses(lambda p: x * (p + 1), n_poses, [x], lambda img, p: img.pow(2).sum())
        expect = 2 * torch.tensor([2.0, -1.0]) * sum((p + 1) ** 2 for p in range(n_poses))
        ok = ok and torch.allclose(gx, expect)
        ret[rank] = bool(ok)
    finally:
        dist.destroy_process_group()


def test_gloo_world_size_2():
    world = 2
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(world, _free_port(), ret), nprocs=world, join=True)
    assert all(ret.get(r) for r in range(world)), dict(ret)


def _tile_worker(rank, world, port, emu_so, out_path):
    """One rank of a REAL sharded render on CPU: the device headers' host build (tools/cpu_emu, test infrastructure) behind the
    C ABI, stripes through rb_scene_set_partition, framebuffer and gradients through the packed gloo all-reduce."""
    import ctypes
    import numpy as np
    from redner_b200 import _lib
    _lib._lib = _lib._bind(ctypes.CDLL(emu_so))  # this process only
    from redner_b200 import redner as rb
    import parity_utils as pu
    import scenes
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        dev = torch.device("cpu")
        sc = scenes.glossy_room(dev, resolution=(26, 22))
        img = rdist.render_tiles(sc, 4, 2, seed=5, rows_per_stripe=4, sampler_type=rb.SamplerType.sobol, device=dev, backend=rb,
                                 use_primary_edge_sampling=True, use_secondary_edge_sampling=True)  # (the boundary-term pick is a pure function
        img.pow(2).sum().backward()                                                                    # of pixel, sample and depth: shardable)
        if rank == 0:
            g = pu.collect_grads(sc)
            np.savez(out_path, image=img.detach().numpy(), **{k: v.numpy() for k, v in g.items()})
    finally:
        dist.destroy_process_group()


def test_gloo_world_size_2_renders_the_same_image_and_gradients_as_one_rank(tmp_path):
    """N > 1 with real rendering, on CPU: two gloo ranks render disjoint stripes of one image (and disjoint shares of the
    primary-edge samples); the all-reduced image must equal the single-rank image bit for bit and every all-reduced gradient
    the single-rank gradient up to summation order."""
    import numpy as np
    import test_device_code_cpu as tdc
    emu = tdc._build()
    outs = {}
    for world in (1, 2):
        path = str(tmp_path / ("w%d.npz" % world))
        mp.spawn(_tile_worker, args=(world, _free_port(), emu, path), nprocs=world, join=True)
        outs[world] = dict(np.load(path))
    a, b = outs[1], outs[2]
    assert np.array_equal(a["image"], b["image"])
    assert set(a) == set(b) and len(a) > 5
    for k in a:
        n = np.linalg.norm(a[k])
        if k != "image" and n > 0:
            assert np.linalg.norm(a[k] - b[k]) / n < 1e-5, k


def _batch_worker(rank, world, port, emu_so, out_path):
    """One rank of the C5 shape on CPU: the rank's share of the camera poses through ONE native scene (api.render_batch ->
    rb_scene_set_camera per view, host build of the device headers behind the C ABI), then one packed all-reduce of the gradients of the
    shared geometry / materials / lights (bench.py --workload c5 under torchrun does this with NCCL)."""
    import ctypes
    import numpy as np
    from redner_b200 import _lib
    _lib._lib = _lib._bind(ctypes.CDLL(emu_so))  # this process only
    from redner_b200 import api, redner as rb
    import parity_utils as pu
    import scenes
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        dev = torch.device("cpu")
        poses = [([0.3, 1.4, -4.5], [0.0, 0.6, 0.0]), ([1.2, 1.1, -4.0], [0.1, 0.5, 0.1]), ([-0.8, 1.8, -4.2], [0.0, 0.7, 0.2]), ([0.0, 2.2, -3.8], [0.0, 0.5, 0.0])]
        mine = list(range(rank, len(poses), world))
        views = [scenes.glossy_room(dev, resolution=(20, 20)) for _ in mine]
        for v, k in zip(views, mine):
            p, l = poses[k]
            v.camera = api.Camera(position=torch.tensor(p), look_at=torch.tensor(l), up=torch.tensor([0.0, 1.0, 0.0]), fov=torch.tensor([40.0]), clip_near=1e-2,
                                  resolution=(20, 20))
            v.shapes, v.materials, v.area_lights = views[0].shapes, views[0].materials, views[0].area_lights
        imgs = api.render_batch(views, 4, 2, [21 + k for k in mine], sampler_type=rb.SamplerType.sobol, device=dev, backend=rb)
        imgs.pow(2).sum().backward()
        g = {k: v for k, v in pu.collect_grads(views[0]).items() if not k.startswith("cam.")}
        keys = sorted(g)
        reduced = rdist.all_reduce_packed([g[k] for k in keys])
        gathered = [None] * world
        dist.all_gather_object(gathered, (mine, imgs.detach().numpy()))
        if rank == 0:
            full = np.zeros((len(poses),) + tuple(imgs.shape[1:]), dtype=np.float32)
            for ids, arr in gathered:
                full[ids] = arr
            np.savez(out_path, images=full, **{k: r.numpy() for k, r in zip(keys, reduced)})
    finally:
        dist.destroy_process_group()


def test_gloo_world_size_2_batch_of_poses_equals_one_rank(tmp_path):
    """The C5 partition (independent poses, no data-path collective, one gradient all-reduce) at world size 2 against one rank: every
    pose's image bit for bit, the summed gradients up to summation order."""
    import numpy as np
    import test_device_code_cpu as tdc
    emu = tdc._build()
    outs = {}
    for world in (1, 2):
        path = str(tmp_path / ("b%d.npz" % world))
        mp.spawn(_batch_worker, args=(world, _free_port(), emu, path), nprocs=world, join=True)
        outs[world] = dict(np.load(path))
    a, b = outs[1], outs[2]
    assert a["images"].shape[0] == 4 and np.array_equal(a["images"], b["images"]) and np.abs(a["images"]).sum() > 0
    assert set(a) == set(b) and len(a) > 4
    for k in a:
        n = np.linalg.norm(a[k])
        if k != "images" and n > 0:
            assert np.linalg.norm(a[k] - b[k]) / n < 1e-5, k
