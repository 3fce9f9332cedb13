"""CPU check of the DEVICE code's arithmetic: the rb_*.cuh headers the sm_100a kernels are built from are compiled
with g++ (tools/cpu_emu: plain loops instead of kernels, host pointers behind the same C ABI) and every golden case
-- images and gradients produced by the unmodified reference -- must be met with the tolerances of the GPU suite.

This is test infrastructure, not a CPU path of the product (redner_b200/ cannot load it, tests/test_abi_cpu.py
pins that); it lets a change to the per-sample code be checked against the reference before a GPU is available.
Launch structure, compaction, sorting, atomics and the lean instantiation are only covered by `-m gpu`.
"""
import hashlib
import os
import shutil
import subprocess
import sys

import pytest

import parity_utils as pu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU_DIR = os.path.join(ROOT, "tools", "cpu_emu")
CSRC = os.path.join(ROOT, "redner_b200", "csrc")


def _source_hash():
    h = hashlib.sha1()
    files = [os.path.join(EMU_DIR, f) for f in ("emu.cpp", "emu_shim.h", "build.sh")]
    files += [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith((".cuh", ".hpp", ".h"))]
    files.append(os.path.join(ROOT, "include", "redner_b200.h"))
    for f in files:
        h.update(open(f, "rb").read())
    return h.hexdigest()[:12]


def _build(flags=""):
    if shutil.which("g++") is None or not os.path.isdir("/usr/local/cuda/include"):
        pytest.skip("needs g++ and the CUDA headers")
    out_dir = os.path.join(ROOT, "tests", "_build")
    os.makedirs(out_dir, exist_ok=True)
    tag = hashlib.sha1((_source_hash() + flags).encode()).hexdigest()[:12]
    so = os.path.join(out_dir, "libredner_b200_emu_%s.so" % tag)
    if not os.path.exists(so):
        env = dict(os.environ, RB_EMU_OUT=so + ".tmp", RB_EMU_OPT="-O1", RB_EMU_FLAGS=flags)
        subprocess.run(["bash", os.path.join(EMU_DIR, "build.sh")], check=True, env=env, timeout=900)
        os.replace(so + ".tmp", so)
    return so


@pytest.fixture(scope="module")
def emulator():
    return _build()


@pytest.fixture(scope="module")
def emulator_lean():
    """The same headers with -DRB_LEAN: environment map, general cameras and G-buffer channels compiled out, as in
    rb_kernels_lean.cu (the instantiation the driver launches for the common configuration)."""
    return _build("-DRB_LEAN")


def _check(so, names):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "emu_check.py"), so] + names, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert [l for l in r.stdout.splitlines() if l.startswith("ok ")] == ["ok " + n for n in names]


def test_device_headers_meet_every_golden_case(emulator):
    _check(emulator, list(pu.CASES))


def test_device_headers_meet_the_gbuffer_goldens(emulator):
    _check(emulator, list(pu.GBUFFER_CASES) + list(pu.SCREEN_CASES))


def test_device_headers_meet_the_boundary_term_statistics(emulator):
    """Secondary-edge (shadow) gradients: mean over seeds against the reference's mean +- standard error, incl. the
    low-sample-count case that pins the reference's strategy coin."""
    _check(emulator, list(pu.STAT_CASES))


def test_batch_of_views_through_one_native_scene(emulator):
    """api.render_batch / rb_scene_set_camera: host logic of the batch path (views share geometry, per view only the camera-dependent
    tables are rebuilt), checked against one full Scene per view; the GPU twin is tests/test_scene_build_gpu.py."""
    _check(emulator, ["batch_of_views"])


def test_lean_instantiation_meets_the_goldens_it_serves(emulator_lean):
    names = [n for n, c in pu.CASES.items() if "channels" not in c and c["scene"] in ("single_triangle", "shadow_blocker", "glossy_room", "nmap_room")]
    assert len(names) >= 7
    _check(emulator_lean, names + ["c2_all_vertices_secondary_stat"])


def test_random_scene_sweep_against_the_live_reference(emulator):
    """tools/fuzz_emu.py on a fixed range of seeds: random cameras / meshes / materials / lamps / options rendered and
    differentiated by the host build of the device headers and compared with the reference's outputs for the same scenes
    (tests/golden/fuzz_reference.npz, written by tests/golden/make_golden.py); nothing may be flagged."""
    golden = os.path.join(ROOT, "tests", "golden", "fuzz_reference.npz")
    r = subprocess.run([sys.executable, "-W", "ignore", os.path.join(ROOT, "tools", "fuzz_emu.py"), emulator, "0", "80", "--golden", golden], capture_output=True,
                       text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    assert r.stdout.strip().splitlines()[-1] == "flagged 0 of 80", "\n".join(l for l in r.stdout.splitlines() if "<<<<" in l or "ERROR" in l)[-3000:]


def test_secondary_edges_sample_by_sample_with_the_reference_streams():
    """a17 without statistics: with the boundary-sample streams indexed like the reference's compacted wavefront
    (-DRB_EMU_REF_STREAMS, possible only in a sequential host build) every secondary-edge gradient equals the reference's."""
    _check(_build("-DRB_EMU_REF_STREAMS"), list(pu.REFSTREAM_CASES))
