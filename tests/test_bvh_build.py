"""SURVEY §8(f1): the BVH build.  The tree decides tie-breaks of the traversal, so both builders must produce THE reference tree:
  * CPU: crloader_build_bvh (the host builder on its own) reproduces, from the triangles of a flat scene, the BVH the scene loader /
    the reference's own loader stored in that scene (node for node, bit for bit);
  * GPU: crgpu_bvh_build (level-synchronous device build, c-ray_b200/csrc/crgpu_bvh_build.cu) equals the host builder bit for bit on
    every mesh of the bundled scenes and on adversarial inputs (ties, duplicates, signed zeros, degenerate boxes, tiny inputs)."""
import os
import subprocess

import numpy as np
import pytest

import crgpu
import crscene
from conftest import GOLDEN, GOLDEN_SCENES, NO_BUNDLED, ROOT


def mesh_inputs(path):
    """[(name, bboxes, centers, stored nodes, stored prims)] for every mesh of a .crscene"""
    import ctypes as C
    flat = crgpu.FlatScene()
    assert crgpu.lib().crscene_load(C.byref(flat), os.fsencode(path)) == 0      # crscene_io.c is part of libcrgpu.so; no device needed
    A = crscene.arrays(flat)
    out = []
    for m, mesh in enumerate(A["meshes"]):
        polys = A["polys"][mesh["poly_offset"]:mesh["poly_offset"] + mesh["poly_count"]]
        bb, ct = crscene.prim_boxes(A["vertices"], polys)
        b = A["bvhs"][mesh["bvh"]]
        nodes = A["bvh_nodes"][b["node_offset"]:b["node_offset"] + b["node_count"]]
        prims = A["prim_indices"][b["prim_offset"]:b["prim_offset"] + b["prim_count"]]
        out.append((f"{os.path.basename(path)}:mesh{m}", bb, ct, nodes, prims))
    return out


def same_tree(a_nodes, a_prims, b_nodes, b_prims):
    assert len(a_nodes) == len(b_nodes), (len(a_nodes), len(b_nodes))
    assert np.array_equal(a_prims, b_prims)
    used = np.uint32(crscene.LEAF_BIT | crscene.COUNT_MASK)        # bit 31 of the reference's bitfield word is never written (bvh.c:37-42)
    assert np.array_equal(a_nodes["first"], b_nodes["first"]) and np.array_equal(a_nodes["count_leaf"] & used, b_nodes["count_leaf"] & used)
    assert np.array_equal(a_nodes["bounds"].view(np.uint32), b_nodes["bounds"].view(np.uint32))      # bit for bit, signed zeros included


def check_tree(nodes, prims, n):
    """structural invariants of any valid result: every primitive in exactly one leaf, children allocated as pairs, boxes nested"""
    assert len(nodes) >= 1 and sorted(prims.tolist()) == list(range(n))
    leaf = (nodes["count_leaf"] & crscene.LEAF_BIT) != 0
    cnt = nodes["count_leaf"] & crscene.COUNT_MASK
    assert len(nodes) == 2 * int(leaf.sum()) - 1
    covered = np.zeros(n, dtype=np.int32)
    for f, c in zip(nodes["first"][leaf], cnt[leaf]):
        covered[f:f + c] += 1
    assert (covered == 1).all()
    for i in np.nonzero(~leaf)[0]:
        for ch in (nodes["first"][i], nodes["first"][i] + 1):
            assert ch > i and ch < len(nodes)
            pb, cb = nodes["bounds"][i], nodes["bounds"][ch]
            if not (nodes["count_leaf"][ch] & crscene.COUNT_MASK) == 0 or not leaf[ch]:      # empty leaves carry the empty box
                assert (cb[0::2] >= pb[0::2]).all() and (cb[1::2] <= pb[1::2]).all()


def synthetic_cases():
    rng = np.random.default_rng(7)

    def boxes(centers, ext):
        c = centers.astype(np.float32)
        e = np.abs(ext).astype(np.float32)
        return np.concatenate([c - e, c + e], axis=1).astype(np.float32), c

    cases = []
    for n in (1, 2, 3, 17, 33, 1000):
        cases.append((f"uniform{n}", *boxes(rng.uniform(-5, 5, (n, 3)), rng.uniform(0, 0.3, (n, 3)))))
    cases.append(("identical_centers_40", *boxes(np.zeros((40, 3)) + 1.5, rng.uniform(0.1, 0.2, (40, 3)))))      # median fallback, nothing splits
    cases.append(("duplicates_500", *boxes(np.repeat(rng.uniform(-1, 1, (50, 3)), 10, axis=0), np.full((500, 3), 0.05))))
    g = np.stack(np.meshgrid(np.arange(-8, 8), np.arange(-8, 8), np.array([0.0, -0.0])), -1).reshape(-1, 3).astype(np.float32)
    ext0 = np.zeros_like(g)
    cases.append(("signed_zero_grid", *boxes(g, ext0)))                                                         # flat boxes, +0 / -0 ties everywhere
    cases.append(("line_2000", *boxes(np.stack([np.linspace(-100, 100, 2000), np.zeros(2000), np.zeros(2000)], 1), np.full((2000, 3), 0.01))))
    cases.append(("clustered_100k", *boxes(np.concatenate([rng.normal(0, 0.01, (50000, 3)), rng.normal(50, 20, (50000, 3))]), rng.uniform(0, 0.05, (100000, 3)))))
    return cases


@pytest.mark.parametrize("name", GOLDEN_SCENES)
def test_host_builder_reproduces_the_scene_bvh(name):
    meshes = mesh_inputs(os.path.join(GOLDEN, name + ".crscene"))
    for label, bb, ct, nodes, prims in meshes:
        got_nodes, got_prims = crscene.build_bvh(bb, ct)
        same_tree(got_nodes, got_prims, nodes, prims)
        check_tree(got_nodes, got_prims, len(bb))


def test_host_builder_on_synthetic_inputs():
    for label, bb, ct in synthetic_cases():
        nodes, prims = crscene.build_bvh(bb, ct)
        check_tree(nodes, prims, len(bb))
    nodes, prims = crscene.build_bvh(np.zeros((0, 6), np.float32), np.zeros((0, 3), np.float32))
    assert len(nodes) == 0


@pytest.mark.gpu
def test_device_builder_equals_host_builder_on_synthetic_inputs():
    for label, bb, ct in synthetic_cases():
        h_nodes, h_prims = crscene.build_bvh(bb, ct)
        d_nodes, d_prims = crscene.build_bvh_gpu(bb, ct)
        same_tree(d_nodes, d_prims, h_nodes, h_prims)
    d_nodes, _ = crscene.build_bvh_gpu(np.zeros((0, 6), np.float32), np.zeros((0, 3), np.float32))
    assert len(d_nodes) == 0


@pytest.mark.gpu
@pytest.mark.parametrize("scene", ["hdr", "scene", "refraction", "venus", "fence"])
def test_device_builder_reproduces_the_bundled_scene_bvhs(scene, bundled_scene):
    """every mesh BVH of the bundled scenes (hdr.json: the 274,243-triangle Venus, 229,087 nodes) — as the host loader builds them,
    the same as the reference's own loader (tests/test_loader.py) — rebuilt on the device: node for node, bit for bit."""
    path = bundled_scene(scene)
    if path is None:
        pytest.skip(NO_BUNDLED)
    for label, bb, ct, nodes, prims in mesh_inputs(path):
        d_nodes, d_prims = crscene.build_bvh_gpu(bb, ct)
        same_tree(d_nodes, d_prims, nodes, prims)


@pytest.mark.gpu
def test_cli_with_device_bvh_renders_the_same_frame(tmp_path):
    """cray_b200 --gpu-bvh: the loader's BVH builds routed to crgpu_bvh_build; the frame must be the host-built scene's, bit for bit."""
    exe = os.path.join(ROOT, "c-ray_b200", "cray_b200")
    refdir = os.path.join(ROOT, "oracle", "_ref")
    if not os.path.exists(os.path.join(refdir, "input", "hdr.json")):
        pytest.skip("oracle/_ref/input missing")
    outs = []
    for extra in ([], ["--gpu-bvh"]):
        f32 = str(tmp_path / f"o{len(outs)}.f32")
        r = subprocess.run([exe, "input/hdr.json", "-d", "160x90", "-s", "8", "-b", "8", "--dump-f32", f32, "-o", str(tmp_path / "o.png"), "-q"] + extra,
                           cwd=refdir, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=300)
        assert r.returncode == 0, r.stdout[-2000:]
        assert "building on the host" not in r.stdout
        outs.append(np.fromfile(f32, dtype=np.float32))
    assert np.array_equal(outs[0].view(np.uint32), outs[1].view(np.uint32))
