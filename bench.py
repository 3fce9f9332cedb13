#!/usr/bin/env python
"""Benchmark of the hot path: pyredner.RenderFunction forward + backward == two redner.render() calls.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2|c3|c4|c5] [--mode tiles|poses|both]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

Workloads (BASELINE.json configs, SURVEY.md section 8d; meshes of C3 - C5 are the reference's own, tests/golden/scene_*.npz):
  c2  (default, the configuration BASELINE.json's metric is quoted on) tests/test_shadow_blocker.py at 512 x 512 x 64 spp, max_bounces 1
  c3  tests/test_teapot_reflectance.py: teapot.xml (15 712 triangles) 512 x 512 x 256 spp, max_bounces 2, SVBRDF + camera-pose gradients
  c4  tests/test_bunny_box.py: bunny_box.xml (14 416 triangles) 1024 x 1024 x 128 spp, max_bounces 5, bunny vertex gradients
  c5  batch: 64 camera poses x teapot 512 x 512 x 64 spp, max_bounces 2 (poses sharded over the ranks, one NCCL gradient all-reduce)
Sobol sampler, primary + secondary edge sampling, loss = sum(img^2) (dense d_image = 2 img), forward seed s / backward seed s + 1000003.
One "step" = one forward render + one backward render == W*H*spp pixel samples through the whole differentiable path tracer
(c5: of every pose).  metric = fwd+bwd megasamples/s = W*H*spp / (t_forward_call + t_backward_call) / 1e6.

  value  whole-job throughput with the scene tensors resident in HBM; CUDA events on the render stream around the two rb_render
         calls (scene construction -- BVH / light tables / edge tree -- is reported separately in config.scene_build_ms, as
         BASELINE.md section 2 prescribes);
  e2e    the same metric through the public API (redner_b200.api.RenderFunction) starting from HOST tensors in pinned memory:
         host->device copies of every scene tensor, scene construction, forward, loss, backward and the device->host read of
         the image, the loss and all gradients are inside the timed region;
  roofline      dominant kernel / stage of the step: algorithmic bytes of SURVEY.md section 8(d) over its CUDA-event duration;
  cpu_baseline  the unmodified reference (oracle/_ref, CPU/Embree) on a bounded sample of the same workload (rank 0, N = 1 only).

--dump-outputs DIR: after the timed steps, rank 0 writes what the last timed step computed -- the image(s) of the forward call
(`image`, poses stacked along a leading axis when a rank renders several) and every gradient the backward call returns (`grad<i>`, i =
position in RenderFunction.backward's output, after the gradient all-reduce) -- as DIR/<name>.npy in float32.  Inputs are seeded, so two
builds can be compared output for output.  Outputs larger than 64 MB in all are cut to a fixed, seeded sample of their elements.

N > 1, one process per GPU.  `tiles` (the partition north_star names; the headline `value`): ONE image split into 4-row stripes
round-robin over the ranks, all-reduce of framebuffer and gradients (strong scaling).  `poses`: every rank renders a full image
(c2 - c4: the workload's own image on every rank, i.e. identical per-GPU work; c5: its share of the 64 distinct poses), one packed gradient
all-reduce (weak scaling, BASELINE config 5 pattern).  By default both are measured at
N > 1 and the weak-scaling result is reported in the extra key "poses".
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402

SEED = 1
ROWS_PER_STRIPE = 4  # tiles mode: 4-row stripes round-robin (at 8 ranks and 512 rows every rank owns 16 stripes spread over the image)
WORKLOADS = {
    "c2": dict(scene="shadow_blocker", res=512, spp=64, mb=1, label="C2 shadow_blocker (tests/test_shadow_blocker.py)"),
    "c3": dict(scene="teapot", res=512, spp=256, mb=2, label="C3 teapot.xml 15712 tris (tests/test_teapot_reflectance.py)"),
    "c4": dict(scene="bunny_box", res=1024, spp=128, mb=5, label="C4 bunny_box.xml 14416 tris (tests/test_bunny_box.py)"),
    "c5": dict(scene="teapot", res=512, spp=64, mb=2, poses=64, label="C5 batch of 64 camera poses x teapot.xml (BASELINE.json configs[4])"),
}


def bytes_per_sample(d_bar, hit_frac, use_primary, use_secondary):
    """Algorithmic bytes per pixel sample after SURVEY.md section 8(d) (fp32 state of every stage functor of the reference,
    counted once per write and once per consuming read), split by the kernel that does that work here:
      k_forward        750 + 1630 d
      k_bwd_trace      750 + 1630 d                     (primal replay)
      k_bwd_secondary  2650 d + 3260 (d - h)            (boundary terms: edge sample + two sub-paths)
      k_bwd_sweep      448 + 1280 d + 610 h             (reverse sweep, first-hit and camera adjoints)
      k_primary_edge   1700 + 3260 d
    d = mean executed bounces per sample (measured by the backward pass), h = measured primary-hit fraction."""
    a = {"k_forward": 750 + 1630 * d_bar, "k_bwd_trace": 750 + 1630 * d_bar, "k_bwd_sweep": 448 + 1280 * d_bar + 610 * hit_frac}
    a["k_bwd_secondary"] = (2650 * d_bar + 3260 * max(0.0, d_bar - hit_frac)) if use_secondary else 0.0
    a["k_primary_edge"] = (1700 + 3260 * d_bar) if use_primary else 0.0
    return a


def timed_builds_ms(builds, n_timed):
    """Mean wall time of the scene builds of the TIMED steps: the first build of a process also loads the build kernels' modules and grows
    the memory pool (reported separately as scene_build_first_ms)."""
    tail = builds[-n_timed:] if n_timed > 0 else builds
    return sum(tail) / max(1, len(tail))


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Write {name: array} as out_dir/<name>.npy in float32.  If they exceed DUMP_BYTES in all, the small arrays are kept whole and
    the larger ones are replaced by the same fixed, seeded sample of their flattened elements (distinct, sorted indices) on every
    run, so that the files of two runs stay comparable element for element."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: np.ascontiguousarray(v, dtype=np.float32) for k, v in arrays.items()}
    left, todo = DUMP_BYTES // 4, sorted(arrays, key=lambda k: arrays[k].size)
    for i, name in enumerate(todo):
        a = arrays[name]
        take = min(a.size, left // (len(todo) - i))
        if take < a.size:
            a = a.ravel()[np.sort(np.random.RandomState(i).choice(a.size, take, replace=False))]
        left -= a.size
        np.save(os.path.join(out_dir, name + ".npy"), a)


def measured_traffic(workload):
    """DRAM bytes per step of each kernel from the committed ncu capture of this build (profiles/r02_<workload>_dram_traffic.json)."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "r02_%s_dram_traffic.json" % workload)))
    except Exception:
        return {}


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons during the timed region (NVML in-process; nvidia-smi as fallback)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.rows = index, False, []

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            bits = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))
            while not self.stop_flag:
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.rows.append([str(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)), str(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))] +
                                 ["Active" if r & b else "Not Active" for _, b in bits])
                time.sleep(0.05)
            return
        except Exception:
            pass
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(self.rows)}


# ------------------------------------------------------------------------------------------------ scenes
def make_scene(wl, device, pose=None):
    """Scene of a workload on `device`.  `pose` (int): camera pose index -- C2: the camera rotated about the scene; teapot: orbit."""
    import scenes
    res = (wl["res"], wl["res"])
    if wl["scene"] == "teapot" and pose is not None:
        return scenes.teapot_pose(device, pose, num_poses=wl.get("poses", 64), resolution=res)
    sc = scenes.SCENES[wl["scene"]](device, resolution=res)
    if pose and wl["scene"] == "shadow_blocker":
        a = 0.05 * pose
        sc.camera.position = torch.tensor([5.0 * math.sin(a), 2.0, -5.0 * math.cos(a)])
    return sc


def scene_tensors(sc):
    """Every tensor of a scene as (owner, attribute, tensor): geometry, textures, light intensities (camera stays on the host)."""
    out = []
    for s in sc.shapes:
        for k in ("vertices", "indices", "uvs", "normals", "uv_indices", "normal_indices", "colors"):
            t = getattr(s, k, None)
            if t is not None:
                out.append((s, k, t))
    for m in sc.materials:
        for k in ("diffuse_reflectance", "specular_reflectance", "roughness", "generic_texture", "normal_map"):
            tex = getattr(m, k, None)
            if tex is not None:
                out.append((tex, "texels", tex.texels))
                out.append((tex, "uv_scale", tex.uv_scale))
    return out


def leaf_params(sc):
    ps = [t for _, _, t in scene_tensors(sc) if t.requires_grad]
    ps += [l.intensity for l in sc.area_lights if l.intensity.requires_grad]
    cam = sc.camera
    ps += [t for t in (cam.position, cam.look_at, cam.up) if t is not None and t.requires_grad]
    return ps


class HostScene:
    """A workload's scene held in PINNED host memory; `to_device()` rebuilds it on the GPU (the per-step H2D of the e2e leg)."""

    def __init__(self, wl, pose=None):
        from redner_b200 import api
        self.api = api
        self.sc = make_scene(wl, torch.device("cpu"), pose)
        self.shapes, self.mats = [], []
        pin = lambda t: t.detach().contiguous().pin_memory()  # noqa: E731
        for s in self.sc.shapes:
            self.shapes.append(({k: pin(getattr(s, k)) for k in ("vertices", "indices", "uvs", "normals", "uv_indices", "normal_indices", "colors")
                                 if getattr(s, k, None) is not None}, s.material_id, s.vertices.requires_grad))
        for m in self.sc.materials:
            texs = {}
            for k in ("diffuse_reflectance", "specular_reflectance", "roughness", "generic_texture", "normal_map"):
                tex = getattr(m, k, None)
                if tex is not None:
                    texs[k] = (pin(tex.texels), pin(tex.uv_scale), tex.texels.requires_grad)
            self.mats.append((texs, m))
        self.h2d_bytes = sum(t.numel() * t.element_size() for d, _, _ in self.shapes for t in d.values()) + \
            sum(a.numel() * a.element_size() + b.numel() * b.element_size() for texs, _ in self.mats for a, b, _ in texs.values())

    def to_device(self, dev):
        api = self.api
        shapes, mats, params = [], [], []
        for d, mid, grad in self.shapes:
            t = {k: v.to(dev, non_blocking=True) for k, v in d.items()}
            if grad:
                t["vertices"].requires_grad_(True)
                params.append(t["vertices"])
            shapes.append(api.Shape(t["vertices"], t["indices"], mid, **{k: v for k, v in t.items() if k not in ("vertices", "indices")}))
        for texs, m in self.mats:
            kw = {}
            for k, (tx, uv, grad) in texs.items():
                tx = tx.to(dev, non_blocking=True)
                if grad:
                    tx.requires_grad_(True)
                    params.append(tx)
                kw[k] = api.Texture(tx, uv.to(dev, non_blocking=True))
            mats.append(api.Material(two_sided=m.two_sided, use_vertex_color=getattr(m, "use_vertex_color", False), **kw))
        lights = []
        for l in self.sc.area_lights:
            inten = l.intensity.detach().clone().requires_grad_(l.intensity.requires_grad)
            if inten.requires_grad:
                params.append(inten)
            lights.append(api.AreaLight(l.shape_id, inten, l.two_sided, l.directly_visible))
        cam = self.sc.camera
        for t in (cam.position, cam.look_at, cam.up):
            if t is not None and t.requires_grad:
                t.grad = None
                params.append(t)
        return api.Scene(cam, shapes, mats, lights), params


# ------------------------------------------------------------------------------------------------ our arm
def run_ours(args, rank, world, local_rank):
    from redner_b200 import api, dist as rdist
    from redner_b200 import redner as rb
    wl = WORKLOADS[args.workload]
    RES, SPP, MB = wl["res"], wl["spp"], wl["mb"]
    dev = torch.device("cuda:%d" % local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        torch.distributed.init_process_group("nccl", device_id=dev)
    st = rb.SamplerType.sobol
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)  # > 126 MB L2
    n_poses = wl.get("poses", 0)
    modes = ["single"] if world == 1 else (["tiles", "poses"] if args.mode == "both" else [args.mode])
    if n_poses:
        modes = ["poses"]  # C5 is a batch of poses by definition
    # poses of this rank.  C5: its share of the 64 distinct poses.  Other workloads, weak mode: every rank renders the workload's own
    # image (pose None) -- weak scaling in the strict sense, per-GPU work identical, so the line isolates the collective; ranks that
    # render DIFFERENT poses (C5) finish at different times and the collective absorbs the skew (see per_rank_compute_ms).
    my_poses = list(range(rank, n_poses, world)) if n_poses else [None]

    def timed_loop(step, steps):
        """W warm-up steps, then K timed steps (L2 flushed before each), barrier + synchronize on both sides, MAX over ranks."""
        for _ in range(args.warmup):
            step()
            flush.zero_()
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()
        times, infos = [], []
        for _ in range(steps):
            flush.zero_()  # evict the previous step's working set from L2
            torch.cuda.synchronize()
            t, info = step()
            times.append(t)
            infos.append(info)
        torch.cuda.synchronize()
        if world > 1:
            torch.distributed.barrier()
        total_ms = sum(times)
        rank_ms = total_ms
        if world > 1:
            tt = torch.tensor([total_ms], device=dev)
            torch.distributed.all_reduce(tt, op=torch.distributed.ReduceOp.MAX)
            total_ms = tt.item()
        return total_ms / steps, rank_ms / steps, infos

    # ---------------- device-resident throughput ----------------
    def make_resident_step(mode):
        scs = [make_scene(wl, dev, pose=p) for p in (my_poses if mode == "poses" else [None])]
        builds = []

        def render_pair(sc):
            """The two rb_render calls of one image, timed with CUDA events on the render stream."""
            for p in leaf_params(sc):
                p.grad = None
            fargs = api.RenderFunction.serialize_scene(sc, SPP, MB, sampler_type=st, device=dev)
            t0 = time.perf_counter()
            c = api.RenderFunction._unpack((SEED, SEED + 1000003), fargs)  # scene construction (BVH, lights, edges, edge tree)
            torch.cuda.synchronize()
            builds.append((time.perf_counter() - t0) * 1e3)
            if mode == "tiles":
                c.scene.set_partition(rank, world, ROWS_PER_STRIPE)
            nch = rb.compute_num_channels(c.channels, c.scene.max_generic_texture_dimension)
            img = torch.zeros(RES, RES, nch, device=dev)
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(6)]
            ev[0].record()
            rb.render(c.scene, c.options, rb.float_ptr(img.data_ptr()), rb.float_ptr(0), None, rb.float_ptr(0), rb.float_ptr(0))
            ev[1].record()
            fwd_stats = c.scene.last_stage_stats()
            if mode == "tiles":  # disjoint stripes: the sum is a gather of the framebuffer
                torch.distributed.all_reduce(img)
            ev[2].record()
            d_img = (2 * img).contiguous()
            ctx = type("Ctx", (), {})()
            ctx.c, ctx.args = c, fargs
            ev[3].record()
            grads = api.RenderFunction.backward(ctx, d_img)
            ev[4].record()
            bwd_stats = c.scene.last_stage_stats()
            tens = [(i, g.to(dev, non_blocking=True)) for i, g in enumerate(grads) if isinstance(g, torch.Tensor)]
            return ev, img, tens, dict(build=c.scene.build_ms(), fwd_k=fwd_stats[0], bwd_k=bwd_stats[0], vertices=bwd_stats[1], hits=bwd_stats[2],
                                       launches=c.scene.last_stats()[0])

        compute_ms = [0.0]
        last = {}  # --dump-outputs: the images and gradients of the latest step

        def step():
            total, acc, info, imgs = 0.0, None, None, []
            for sc in scs:
                ev, img, tens, info = render_pair(sc)
                grad_ids = [i for i, _ in tens]
                acc = [g for _, g in tens] if acc is None else [a + b for a, (_, b) in zip(acc, tens)]
                if args.dump_outputs:
                    imgs.append(img)
                e5 = ev[5]
                if world > 1 and sc is scs[-1]:  # one packed gradient all-reduce per step (tiles: partial sums; poses: data parallel)
                    acc = rdist.all_reduce_packed(acc)
                e5.record()
                torch.cuda.synchronize()
                fwd, comm_f, bwd, comm_b = ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2]), ev[3].elapsed_time(ev[4]), ev[4].elapsed_time(e5)
                total += fwd + bwd + (comm_f + comm_b if world > 1 else 0.0)
                compute_ms[0] += fwd + bwd
                info.update(fwd_ms=fwd, bwd_ms=bwd, comm_ms=(comm_f + comm_b) if world > 1 else 0.0)
            if args.dump_outputs:
                last["image"] = imgs[0] if len(imgs) == 1 else torch.stack(imgs)
                last.update(("grad%d" % i, g) for i, g in zip(grad_ids, acc))
            return total, info
        return step, builds, compute_ms, last

    results = {}
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    for mode in modes:
        step, builds, compute_ms, last = make_resident_step(mode)
        ms, rank_ms, infos = timed_loop(step, args.steps)
        if args.dump_outputs and rank == 0 and mode == modes[0]:
            dump_outputs(args.dump_outputs, {k: v.detach().cpu().numpy() for k, v in last.items()})
        imgs_per_step = (len(my_poses) if mode == "poses" else 1)
        job_imgs = (n_poses if n_poses else world) if mode == "poses" else 1
        per_rank, per_rank_compute = None, None
        if world > 1:  # per-rank step times with and without the collectives: rank skew vs collective latency
            tt = torch.zeros(2, world, device=dev)
            tt[0, rank] = rank_ms
            tt[1, rank] = compute_ms[0] / (args.steps + args.warmup)
            torch.distributed.all_reduce(tt)
            per_rank = [round(x, 3) for x in tt[0].tolist()]
            per_rank_compute = [round(x, 3) for x in tt[1].tolist()]
        results[mode] = dict(ms=ms, value=job_imgs * RES * RES * SPP / (ms * 1e-3) / 1e6, infos=infos, builds=builds, per_rank_ms=per_rank, per_rank_compute_ms=per_rank_compute,
                             imgs_per_rank=imgs_per_step)

    # ---------------- end to end from pinned host memory (e2e) ----------------
    main_mode = modes[0]
    hosts = [HostScene(wl, pose=p) for p in (my_poses if main_mode == "poses" else [None])]
    h2d = hosts[0].h2d_bytes if n_poses else sum(h.h2d_bytes for h in hosts)
    d2h_box = [0]

    def step_e2e():
        outs, acc = [], None
        if n_poses:
            # C5: ONE host->device copy and ONE native scene for all poses of this rank (api.render_batch / rb_scene_set_camera:
            # per pose only the camera-dependent tables are rebuilt, on the device)
            scn, params = hosts[0].to_device(dev)
            views = []
            for h in hosts:
                v = api.Scene(h.sc.camera, scn.shapes, scn.materials, scn.area_lights)
                for t in (v.camera.position, v.camera.look_at, v.camera.up):
                    if t is not None and t.requires_grad:
                        t.grad = None
                        if all(t is not q for q in params):
                            params.append(t)
                views.append(v)
            imgs = api.render_batch(views, SPP, MB, [SEED + k for k in range(len(views))], sampler_type=st, device=dev)
            loss = imgs.pow(2).sum()
            loss.backward()
            outs += [imgs.detach().to("cpu", non_blocking=True), loss.detach().cpu()]
            acc = [p.grad for p in params]
        else:
            for h in hosts:
                scn, params = h.to_device(dev)
                if main_mode == "tiles":
                    img = rdist.render_tiles(scn, SPP, MB, SEED, rows_per_stripe=ROWS_PER_STRIPE, sampler_type=st, device=dev)
                else:
                    img = api.RenderFunction.apply(SEED, *api.RenderFunction.serialize_scene(scn, SPP, MB, sampler_type=st, device=dev))
                loss = img.pow(2).sum()
                loss.backward()
                outs += [img.detach().to("cpu", non_blocking=True), loss.detach().cpu()]
                gs = [p.grad for p in params]
                acc = gs if acc is None else [a + b.to(a.device) for a, b in zip(acc, gs)]
        if world > 1 and main_mode == "poses":
            cuda_g = [g.to(dev) for g in acc]
            acc = rdist.all_reduce_packed(cuda_g)
        outs += [g.cpu() for g in acc]
        torch.cuda.synchronize()
        d2h_box[0] = sum(o.numel() * o.element_size() for o in outs)
        return 0.0, None

    for _ in range(max(1, args.warmup // 2)):
        step_e2e()
    torch.cuda.synchronize()
    if world > 1:
        torch.distributed.barrier()
    e2e_steps = max(1, min(args.steps, 5 if n_poses else args.steps))
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        step_e2e()
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / e2e_steps
    if world > 1:
        tt = torch.tensor([e2e_ms], device=dev)
        torch.distributed.all_reduce(tt, op=torch.distributed.ReduceOp.MAX)
        e2e_ms = tt.item()
    main = results[main_mode]
    job_imgs_main = (n_poses if n_poses else world) if main_mode == "poses" else 1
    e2e_value = job_imgs_main * RES * RES * SPP / (e2e_ms * 1e-3) / 1e6
    if rank == 0:
        clocks.stop_flag = True
        clocks.join(timeout=2)
    if rank != 0:
        return

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_gbs, peak_src = (peaks["hbm_gbs"], "measured (MEASURED_PEAKS.json)") if "hbm_gbs" in peaks else (6650.0, "fallback (B200_PROFILING.md)")
    info = next((i for i in reversed(main["infos"]) if i), None)
    cfg = {"workload": "%s %dx%dx%dspp max_bounces=%d sobol, primary+secondary edge sampling, loss=sum(img^2)" % (wl["label"], RES, RES, SPP, MB),
           "parallelism": "single GPU" if world == 1 else {"tiles": "%d ranks, one image in %d-row stripes round-robin, NCCL all-reduce of framebuffer + gradients" % (world, ROWS_PER_STRIPE),
                                                           "poses": "%d ranks, %d image(s) per rank, one NCCL gradient all-reduce" % (world, main["imgs_per_rank"])}[main_mode],
           "l2": "256 MB flush between timed steps", "scene_build_ms": timed_builds_ms(main["builds"], args.steps * main["imgs_per_rank"]), "scene_build_first_ms": main["builds"][0] if main["builds"] else None,
           "e2e": "pinned host tensors -> H2D -> scene build -> forward -> loss -> backward -> D2H of image, loss and every gradient (host clock)"}
    roofline = None
    if info:
        n_samples = RES * RES * SPP / (world if main_mode == "tiles" else 1)
        d_bar, hit_frac = info["vertices"] / n_samples, info["hits"] / n_samples
        alg = bytes_per_sample(d_bar, hit_frac, True, True)
        kms = {"k_forward": info["fwd_k"]["k_forward"], **{k: v for k, v in info["bwd_k"].items() if k in alg and k != "k_forward"}}
        tr = measured_traffic(args.workload)
        traffic = dict(tr.get("dram_bytes_per_step", {}))
        for stage, names in {"k_bwd_secondary": ("k_bwd_sec_pick", "k_bwd_sec_shade", "k_sec_offsets", "k_sec_scatter"), "k_primary_edge": ("k_primary_edge", "k_prim_keys")}.items():
            if any(n in traffic for n in names):
                traffic[stage] = sum(traffic.get(n, 0.0) for n in names)
        per_kernel = {k: {"ms": kms[k], "algorithmic_GB": alg[k] * n_samples / 1e9, "achieved_GBps": alg[k] * n_samples / (kms[k] * 1e-3) / 1e9,
                          "frac": alg[k] * n_samples / (kms[k] * 1e-3) / 1e9 / peak_gbs,
                          "dram_GB_measured": (traffic[k] / 1e9 if k in traffic else None)} for k in kms if kms[k] > 0}
        dom = max(per_kernel, key=lambda k: per_kernel[k]["ms"])
        achieved = per_kernel[dom]["achieved_GBps"]
        roofline = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak_gbs, "unit": "GB/s", "frac": achieved / peak_gbs,
                    "traffic": traffic.get(dom), "traffic_source": tr.get("source"), "peak_source": peak_src, "algorithmic_bytes_per_sample": alg[dom],
                    "kernel_ms": kms[dom], "mean_bounces_per_sample": d_bar, "primary_hit_fraction": hit_frac, "per_kernel": per_kernel,
                    "note": "achieved = SURVEY.md 8(d) algorithmic bytes of the dominant kernel per step / its CUDA-event time summed over the "
                            "step's band launches; traffic = dram read+write bytes of those launches (ncu, profiles/).  The kernels keep the "
                            "reference's per-stage state in registers, so DRAM traffic is far below the algorithmic bytes: they are "
                            "issue/latency bound (DESIGN.md section 3), the HBM fraction is the contract's metric, not the limiter"}
        cfg["kernel_ms"] = {"k_forward": info["fwd_k"]["k_forward"], **{k: v for k, v in info["bwd_k"].items() if k != "k_forward"}}
        cfg["scene_build_detail_ms"] = info["build"]
        cfg["fwd_ms"], cfg["bwd_ms"], cfg["comm_ms"] = info["fwd_ms"], info["bwd_ms"], info["comm_ms"]
        # SURVEY.md section 8(d): forward-only and backward-only ("grad") rates of this rank's samples, from the two render calls
        cfg["fwd_msamples_per_s"] = n_samples / (info["fwd_ms"] * 1e-3) / 1e6
        cfg["grad_msamples_per_s"] = n_samples / (info["bwd_ms"] * 1e-3) / 1e6
    if main["per_rank_ms"]:
        cfg["per_rank_step_ms"] = main["per_rank_ms"]
        cfg["per_rank_compute_ms"] = main["per_rank_compute_ms"]  # the two rb_render calls only (without the collectives)
    metric = "fwd+bwd megasamples/s at %dx%dx%dspp" % (RES, RES, SPP)
    out = {"metric": metric, "value": main["value"], "unit": "Msamples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": main["ms"], "higher_is_better": True, "scaling": "weak" if main_mode == "poses" else "strong", "vs_baseline": None, "dtype": "f32",
           "data": "synthetic", "config": cfg, "clocks": clocks.summary(),
           "e2e": {"value": e2e_value, "unit": "Msamples/s", "ms_per_step": e2e_ms, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h_box[0]},
           "gpu_launches": (info["launches"] + 1) * args.steps * main["imgs_per_rank"] if info else 0, "roofline": roofline}
    for mode in modes[1:]:
        r = results[mode]
        i2 = next((i for i in reversed(r["infos"]) if i), None)
        out[mode] = {"value": r["value"], "unit": "Msamples/s", "ms_per_step": r["ms"], "scaling": "weak" if mode == "poses" else "strong",
                     "per_rank_step_ms": r["per_rank_ms"], "per_rank_compute_ms": r["per_rank_compute_ms"], "fwd_ms": i2 and i2["fwd_ms"], "bwd_ms": i2 and i2["bwd_ms"], "comm_ms": i2 and i2["comm_ms"],
                     "note": "every rank renders the workload's image (identical per-GPU work); one packed NCCL gradient all-reduce per step"}
    if world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline(args.workload, budget_s=20.0)
    print(json.dumps(out))


# ------------------------------------------------------------------------------------------------ reference arm / CPU baseline
REF_WORKER = r'''
import json, os, sys, time
ROOT = sys.argv[1]
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests")); sys.path.insert(0, os.path.join(ROOT, "oracle"))
import torch
import bench, ref_loader
from redner_b200 import api
ref = ref_loader.load()
wl = dict(bench.WORKLOADS[sys.argv[2]])
res, spp, reps = int(sys.argv[3]), int(sys.argv[4]), int(sys.argv[5])
wl["res"] = res
dev = torch.device("cpu")
out = []
for _ in range(reps):
    sc = bench.make_scene(wl, dev, pose=0 if wl.get("poses") else None)
    fargs = api.RenderFunction.serialize_scene(sc, spp, wl["mb"], sampler_type=ref.SamplerType.sobol, device=dev, backend=ref)
    c = api.RenderFunction._unpack((bench.SEED, bench.SEED + 1000003), fargs)
    nch = ref.compute_num_channels(c.channels, c.scene.max_generic_texture_dimension)
    img = torch.zeros(res, res, nch)
    t0 = time.perf_counter()
    ref.render(c.scene, c.options, ref.float_ptr(img.data_ptr()), ref.float_ptr(0), None, ref.float_ptr(0), ref.float_ptr(0))
    t1 = time.perf_counter()
    ctx = type("Ctx", (), {})()
    ctx.c, ctx.args = c, fargs
    api.RenderFunction.backward(ctx, (2 * img).contiguous())
    t2 = time.perf_counter()
    out.append([t1 - t0, t2 - t1])
print("REF_TIMES " + json.dumps(out))
'''


def reference_steps(workload, res, spp, reps, threads=None, timeout=3000):
    """fwd / bwd seconds of `reps` fwd+bwd steps of the unmodified reference (CPU/Embree) in a subprocess, optionally pinned to the first
    `threads` cores with taskset (its worker pool sizes itself by std::thread::hardware_concurrency(), src/parallel.cpp:228-235)."""
    cmd = [sys.executable, "-W", "ignore", "-c", REF_WORKER, ROOT, workload, str(res), str(spp), str(reps)]
    if threads:
        cmd = ["taskset", "-c", "0-%d" % (threads - 1)] + cmd
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout)
    for line in r.stdout.splitlines():
        if line.startswith("REF_TIMES "):
            return json.loads(line[len("REF_TIMES "):])
    raise RuntimeError("reference worker failed: " + r.stderr[-500:])


def reference_available():
    return os.path.isdir(os.path.join(ROOT, "oracle", "_ref")) and any(f.startswith("redner") and f.endswith(".so") for f in os.listdir(os.path.join(ROOT, "oracle", "_ref")))


def best_thread_count(workload, cores):
    """The reference's backward pass is bound by contended compare-exchange atomics (BASELINE.md section 3): more threads can be slower.
    Probe a small sample at 1 / 8 / 16 / 32 / all cores and return {threads: Msamples/s}."""
    probe = {}
    res, spp = 64, 4
    for th in sorted(set(t for t in (1, 8, 16, 32, cores) if t <= cores)):
        try:
            (f, b), = reference_steps(workload, res, spp, 1, threads=th, timeout=600)
            probe[th] = res * res * spp / (f + b) / 1e6
        except Exception:
            pass
    return probe


def pick_sample(wl, rate_msps, budget_s):
    """The largest (res, spp) sample of the workload that costs about budget_s seconds per step at `rate_msps`."""
    full = (wl["res"], wl["spp"])
    cands = [full] + [(r, s) for r in (wl["res"], wl["res"] // 2, wl["res"] // 4, 64) for s in (wl["spp"], 64, 16, 8, 4) if r >= 64 and s <= wl["spp"]]
    cands = sorted(set(cands), key=lambda c: -c[0] * c[0] * c[1])
    for res, spp in cands:
        if res * res * spp / (rate_msps * 1e6) <= budget_s:
            return res, spp
    return 64, 4


def cpu_baseline(workload, budget_s):
    cores = os.cpu_count() or 1
    if not reference_available():
        return {"value": None, "unit": "Msamples/s", "cores": cores, "kind": "reference", "sample": "unavailable: oracle/_ref not built"}
    wl = WORKLOADS[workload]
    probe = best_thread_count(workload, cores)
    th = max(probe, key=probe.get)
    res, spp = pick_sample(wl, probe[th], budget_s)
    (f, b), = reference_steps(workload, res, spp, 1, threads=th)
    return {"value": res * res * spp / (f + b) / 1e6, "unit": "Msamples/s", "cores": th, "kind": "reference",
            "sample": "%s %dx%dx%dspp (same scene, sampler, edge sampling and loss%s), fwd %.2fs bwd %.2fs, %d of %d host threads (best of the probe)" %
                      (wl["label"], res, res, spp, "" if (res, spp) == (wl["res"], wl["spp"]) else "; reduced size", f, b, th, cores),
            "fwd_s": f, "bwd_s": b, "thread_probe_msamples_per_s_64x64x4": {str(k): round(v, 4) for k, v in probe.items()}}


def run_reference(args, rank, world):
    if rank != 0:
        return
    if not reference_available():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref not built"}))
        return
    wl = WORKLOADS[args.workload]
    cores = os.cpu_count() or 1
    probe = best_thread_count(args.workload, cores)
    th = max(probe, key=probe.get)
    n = max(1, args.steps + args.warmup)
    budget = max(2.0, float(os.environ.get("RB_REF_TOTAL_S", "180")) / n)  # the whole --steps K --warmup W run stays within a few minutes
    res, spp = pick_sample(wl, probe[th], budget)
    same = (res, spp) == (wl["res"], wl["spp"])
    ts = reference_steps(args.workload, res, spp, n, threads=th)[args.warmup:]
    f = sum(t[0] for t in ts) / len(ts)
    b = sum(t[1] for t in ts) / len(ts)
    v = res * res * spp / (f + b) / 1e6
    # one step of the FULL configuration next to the bounded sample, when the sample's rate says it fits in ~2 minutes
    full = None
    if not same and wl["res"] * wl["res"] * wl["spp"] / (v * 1e6) <= float(os.environ.get("RB_REF_FULL_STEP_MAX_S", "100")):
        try:
            (ff, fb), = reference_steps(args.workload, wl["res"], wl["spp"], 1, threads=th)
            full = {"fwd_s": ff, "bwd_s": fb, "value": wl["res"] * wl["res"] * wl["spp"] / (ff + fb) / 1e6, "unit": "Msamples/s", "threads": th}
        except Exception:
            pass
    sample = "%s %dx%dx%dspp per step (%s), fwd %.2fs bwd %.2fs, %d of %d host threads (fastest of the probe %s)" % (
        wl["label"], res, res, spp, "the full configuration" if same else "bounded sample of the %dx%dx%d workload" % (wl["res"], wl["res"], wl["spp"]), f, b, th, cores,
        {k: round(x, 3) for k, x in probe.items()})
    print(json.dumps({"impl": "reference", "metric": "fwd+bwd megasamples/s at %dx%dx%dspp" % (wl["res"], wl["res"], wl["spp"]), "value": v, "unit": "Msamples/s",
                      "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": (f + b) * 1e3, "higher_is_better": True, "scaling": "strong",
                      "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                      "config": {"workload": "%s %dx%dx%dspp max_bounces=%d sobol, primary+secondary edge sampling, loss=sum(img^2)" % (wl["label"], wl["res"], wl["res"], wl["spp"], wl["mb"]),
                                 "sample": sample, "same_config": same, "full_config_step": full, "parallelism": "reference CPU/Embree path, %d host threads" % th},
                      "cpu_baseline": {"value": v, "unit": "Msamples/s", "cores": th, "kind": "reference", "sample": sample},
                      "e2e": {"value": v, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--mode", default="both", choices=["both", "tiles", "poses"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's image and gradients to DIR/<name>.npy (float32); --impl ours only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank, world, local_rank = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device visible; the redner_b200 render path has no CPU fallback "
                         "(use --impl reference for the CPU baseline)")
    run_ours(args, rank, world, local_rank)
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
