"""Host half of crgpu_scene_create on the CPU, against a stub CUDA runtime (tests/stub/, test tooling only).

crgpu_scene_create validates the flat scene and re-lays it out for the kernels (BFS-ordered 64-byte pair nodes, triangles
packed in leaf order with precomputed edges and normals, per-polygon shading records) on several host threads.  The
kernels' parity with the reference rests on those bytes, so they are pinned here: the running FNV-1a checksum of the big
uploads must not depend on the number of host threads, and malformed scenes must be rejected, not crash."""
import os
import random
import re
import subprocess

import pytest

from conftest import ROOT, GOLDEN, GOLDEN_SCENES, GOLDEN_FLAT, NO_BUNDLED

PKG = os.path.join(ROOT, "c-ray_b200")


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    objs = [os.path.join(PKG, "build", n) for n in ("crgpu_api.o", "crgpu_trace.o", "crgpu_shade.o")]
    if not all(os.path.exists(o) for o in objs):
        pytest.skip("c-ray_b200/build/*.o not present (built by nvcc in build())")
    d = tmp_path_factory.mktemp("stub")
    exe = str(d / "create_harness")
    stub = os.path.join(ROOT, "tests", "stub")
    subprocess.run(["gcc", "-O2", "-c", "-o", str(d / "stub.o"), os.path.join(stub, "cudart_stub.c")], check=True)
    subprocess.run(["gcc", "-O2", "-c", "-I" + os.path.join(ROOT, "include"), "-o", str(d / "h.o"), os.path.join(stub, "create_harness.c")], check=True)
    subprocess.run(["gcc", "-O2", "-c", "-o", str(d / "io.o"), os.path.join(PKG, "host", "crscene_io.c")], check=True)
    subprocess.run(["g++", "-o", exe, str(d / "h.o")] + objs + [str(d / "io.o"), str(d / "stub.o"), "-lpthread"], check=True)
    return exe


def uploads(exe, scene, threads):
    """(slab bytes, FNV-1a of the prepared slab): everything crgpu_scene_create_prepared copies to the device except the two
    small tables that carry device pointers (texture table, DevScene), which are patched per device."""
    env = dict(os.environ, CRGPU_HOST_THREADS=str(threads))
    r = subprocess.run([exe, scene], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=env, timeout=120)
    assert "create rc=0" in r.stdout, r.stdout + r.stderr[-500:]
    m = re.search(r"slab (\d+) bytes sum ([0-9a-f]{16})", r.stdout)
    return int(m.group(1)), m.group(2)


@pytest.mark.parametrize("name", GOLDEN_FLAT)
def test_upload_bytes_do_not_depend_on_host_threads(harness, name):
    scene = os.path.join(GOLDEN, name + ".crscene")
    a, b, c = uploads(harness, scene, 1), uploads(harness, scene, 3), uploads(harness, scene, 8)
    assert a[0] >= 13 * 256 and a == b == c


def test_big_scene_threaded_repack_is_deterministic(harness, bundled_scene):
    scene = bundled_scene("hdr")
    if scene is None:
        pytest.skip(NO_BUNDLED)
    a, b = uploads(harness, scene, 1), uploads(harness, scene, 8)
    assert a == b
    # PackedTri + ShadePoly + PairNode sections of hdr.json (274,245 triangles, 114,552 internal nodes) plus 23 MB of texels
    assert a[0] > 274245 * 48 + 274245 * 80 + 114552 * 64 + 20 * 2 ** 20


@pytest.mark.parametrize("name", ["g_legacy", "g_f4"])
def test_malformed_scenes_are_rejected_not_crashing(harness, tmp_path, name):
    """random byte damage in the array sections (indices, counts, node kinds and operand indices — g_f4 carries the math / vecmath /
    fresnel / combine graphs of the complete interpreter): crgpu_prepare must answer with an error code or accept, never crash"""
    src = open(os.path.join(GOLDEN, name + ".crscene"), "rb").read()
    rng = random.Random(3)
    rejected = 0
    for i in range(150):
        b = bytearray(src)
        for _ in range(rng.randrange(1, 4)):
            b[rng.randrange(16 + 400, len(b))] = rng.randrange(256)          # array sections: indices, counts inside records
        p = tmp_path / "c.crscene"
        p.write_bytes(bytes(b))
        r = subprocess.run([harness, str(p)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=60)
        assert r.returncode == 0 and "create rc=" in r.stdout, (i, r.returncode)    # never a crash
        rejected += "rc=0" not in r.stdout
    assert rejected > 20
