#!/usr/bin/env python3
"""What the unmodified reference produced, stored so that the tests compare against it without the reference.

tests/golden/reference.json holds
  exports  per scene: the reference loader's flat scene (oracle/ref_harness.c `export`) as digests of its header and of
           each array, after the tolerances test_loader.py documents (prefs.thread_count dropped, the unused bits of
           interior BVH nodes cleared, vertex/normal/texcoord slots no polygon reaches left out);
  frames   per render configuration: SHA-256 of the strict reference's fp32 framebuffer bits.
tests/golden/full_config_samples.npz holds a fixed sample of pixels of the full-size frames of BASELINE.json.

Run this file (`python tests/reference_golden.py`) where oracle/_ref/ is built to regenerate both; it runs the
reference binaries: about a CPU-minute, and with `--full` the full-size frames too (tens of CPU-minutes each).
"""
import hashlib
import json
import os
import shutil
import subprocess
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for _p in (HERE, os.path.join(ROOT, "c-ray_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import crgpu    # noqa: E402
import crscene  # noqa: E402

GOLDEN_JSON = os.path.join(HERE, "golden", "reference.json")
FULL_SAMPLES = os.path.join(HERE, "golden", "full_config_samples.npz")
REF_DIR = os.path.join(ROOT, "oracle", "_ref")
REF = os.path.join(REF_DIR, "cray_ref_strict")
BUNDLED = ["hdr", "scene", "refraction", "venus", "alphanode", "fence", "glowmetal", "statues", "uvsphere"]
# (scene, W, H, spp, bounces) of the reference framebuffers the tests compare against (bounces 0 = the JSON's own limit)
FRAMES = [("hdr", 96, 54, 4, 32), ("scene", 80, 50, 4, 4), ("refraction", 64, 36, 2, 512), ("venus", 40, 64, 4, 25),
          ("hdr", 240, 135, 16, 32), ("scene", 320, 200, 16, 4), ("refraction", 240, 135, 8, 512), ("venus", 100, 160, 16, 25),
          ("alphanode", 96, 60, 8, 0), ("fence", 96, 60, 8, 0), ("glowmetal", 96, 60, 8, 0), ("statues", 96, 60, 8, 0),
          ("uvsphere", 96, 60, 8, 0), ("hdr", 1920, 1080, 2, 32), ("venus", 2560, 1600, 1, 25), ("refraction", 1920, 1080, 1, 512)]
# BASELINE.json configurations at full size whose reference frames are sampled into FULL_SAMPLES
FULL = [("hdr", 1920, 1080, 1000, 32), ("refraction", 1920, 1080, 64, 512), ("venus", 2560, 1600, 32, 25)]
SAMPLE_PIXELS = 4096
# the glass total-internal-reflection pixel of tests/test_oracle.py and the block around it (x0, y0, x1, y1, y counted upwards)
TIR_BLOCK = (160, 764, 172, 772)


def frame_key(name, W, H, spp, b):
    return f"{name}_{W}x{H}x{spp}_b{b}"


def frame_digest(img):
    return hashlib.sha256(np.ascontiguousarray(img, dtype=np.float32).tobytes()).hexdigest()


def sample_index(W, H, n=SAMPLE_PIXELS):
    """A fixed spread of n pixel indices (row-major, top row first) over a W x H frame."""
    return (np.arange(n, dtype=np.int64) * 1000003 + 7919) % (W * H)


def _h(b):
    return hashlib.sha256(b).hexdigest()[:16]


def _indexed(A, key):
    """the slots of vertices / normals / texcoords that some polygon indexes"""
    field = {"vertices": "v", "normals": "n", "texcoords": "t"}[key]
    idx = np.unique(A["polys"][field])
    return idx[(idx >= 0) & (idx < len(A[key]))]


def scene_digests(scene):
    """Digests of a FlatScene under the loader tests' tolerances."""
    head = {n: int(getattr(scene, n)) for n, _ in crgpu.FlatScene._fields_
            if n not in ("prefs", "camera", "owner") and n not in [s[0] for s in crscene._SECTIONS]}
    head.update({"prefs." + n: int(getattr(scene.prefs, n)) for n, _ in type(scene.prefs)._fields_ if n != "thread_count"})
    out = {"header": _h(json.dumps(head, sort_keys=True).encode()), "camera": _h(bytes(scene.camera))}
    A = crscene.arrays(scene)
    for key, a in A.items():
        if key == "bvh_nodes":
            a = a.copy()
            leaf = (a["count_leaf"] & crscene.LEAF_BIT) != 0
            a["count_leaf"] = np.where(leaf, a["count_leaf"] & (crscene.COUNT_MASK | crscene.LEAF_BIT), 0)
        elif key in ("vertices", "normals", "texcoords"):
            a = np.ascontiguousarray(a[_indexed(A, key)])
        out[key] = _h(a.tobytes())
    return out


def golden():
    with open(GOLDEN_JSON) as f:
        return json.load(f)


def assert_scene_matches(scene, digests):
    """The loader's scene against a stored reference export."""
    got = scene_digests(scene)
    differ = sorted(k for k in digests if got.get(k) != digests[k])
    assert not differ, f"differs from the reference's export in: {differ}"


# ------------------------------------------------------------------------------------------------ regeneration
def _export_entry(mine_path_json, ref_crscene, cwd):
    """digests of the reference export, checked against the loader's scene for the same input"""
    import test_loader as TL
    old = os.getcwd()
    os.chdir(cwd)
    try:
        mine = crscene.load_json(mine_path_json)
    finally:
        os.chdir(old)
    ref = TL.load_crscene(ref_crscene)
    TL.assert_same_scene(mine, ref)            # the loader agrees with the reference under the documented tolerances
    digests = scene_digests(ref)
    # the digests leave no room for the reference's uninitialised vertex slots (the g_legacy case): such a scene needs the export itself
    assert scene_digests(mine) == digests
    crscene.free(mine)
    return digests


def _ref(args, cwd, timeout=3600):
    r = subprocess.run([REF] + args, cwd=cwd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, errors="replace",
                       timeout=timeout)
    return r.returncode, r.stdout


def regenerate(full=False):
    import tempfile
    import random
    import test_loader as TL
    assert os.path.exists(REF), "oracle/_ref/cray_ref_strict is missing: build() where the reference sources are present"
    out = {"exports": {}, "frames": {}}
    tmp = tempfile.mkdtemp(prefix="cray_golden_")
    threads = str(os.cpu_count() or 1)
    for name in BUNDLED:
        p = os.path.join(tmp, name + ".crscene")
        rc, log = _ref(["export", os.path.join("input", name + ".json"), "0", "0", "0", "0", p], REF_DIR)
        assert rc == 0, log[-2000:]
        out["exports"]["bundled/" + name] = _export_entry(os.path.join("input", name + ".json"), p, REF_DIR)
        os.remove(p)
    for name, W, H, spp, b in FRAMES:
        p = os.path.join(tmp, "f.f32")
        rc, log = _ref(["render", os.path.join("input", name + ".json"), str(W), str(H), str(spp), str(b), threads, "0", "0", p], REF_DIR)
        assert rc == 0, log[-2000:]
        out["frames"][frame_key(name, W, H, spp, b)] = frame_digest(np.fromfile(p, dtype=np.float32))
    for seed in range(TL.FUZZ_SEEDS):
        d = os.path.join(tmp, "fuzz%d" % seed)
        os.makedirs(d)
        TL.write_fuzz_scene(seed, d)
        rc, log = _ref(["export", "fuzz.json", "0", "0", "0", "0", "ref.crscene"], d, 120)
        assert rc == 0, log[-2000:]
        out["exports"]["fuzz/%d" % seed] = _export_entry("fuzz.json", os.path.join(d, "ref.crscene"), d)
    for seed in range(TL.ODD_SEEDS):
        d = os.path.join(tmp, "odd%d" % seed)
        os.makedirs(d)
        if not TL.write_odd_scene(seed, d):
            continue
        rc, log = _ref(["export", "s.json", "0", "0", "0", "0", "ref.crscene"], d, 60)
        assert rc == 0, (seed, log[-500:])
        out["exports"]["odd/%d" % seed] = _export_entry("s.json", os.path.join(d, "ref.crscene"), d)
    d = os.path.join(tmp, "big")
    os.makedirs(d)
    TL._big_scene(d, random.Random(5))
    rc, log = _ref(["export", "big.json", "0", "0", "0", "0", "ref.crscene"], d, 300)
    assert rc == 0, log[-2000:]
    out["exports"]["big"] = _export_entry("big.json", os.path.join(d, "ref.crscene"), d)
    d = os.path.join(tmp, "texfail")
    os.makedirs(d)
    TL.write_texture_fallback_scene(d)
    rc, _ = _ref(["export", "s.json", "0", "0", "0", "0", "ref.crscene"], d, 60)
    # the reference aborts on this input (textureloader.c:78-84 frees a texture that lives in the node pool): nothing to store then
    out["exports"]["texture_fallback"] = _export_entry("s.json", os.path.join(d, "ref.crscene"), d) if rc == 0 else None
    with open(GOLDEN_JSON, "w") as f:
        json.dump(out, f, indent=0, sort_keys=True)
        f.write("\n")
    if full:
        samples = {}
        for name, W, H, spp, b in FULL:
            p = os.path.join(tmp, "full.f32")
            rc, log = _ref(["render", os.path.join("input", name + ".json"), str(W), str(H), str(spp), str(b), threads, "0", "0", p],
                           REF_DIR, 6 * 3600)
            assert rc == 0, log[-2000:]
            add_full_sample(samples, (name, W, H, spp, b), np.fromfile(p, dtype=np.float32).reshape(H, W, 3))
        np.savez(FULL_SAMPLES, **samples)
    shutil.rmtree(tmp)

def add_full_sample(samples, config, img):
    """the stored part of a full-size reference frame: its pixels at sample_index, and for hdr 1000 spp the TIR block"""
    name, W, H, spp, b = config
    samples[frame_key(*config)] = img.reshape(-1, 3)[sample_index(W, H)]
    if (name, W, H, spp) == ("hdr", 1920, 1080, 1000):
        x0, y0, x1, y1 = TIR_BLOCK
        samples["tir_block"] = img[H - y1:H - y0, x0:x1]


if __name__ == "__main__":
    regenerate(full="--full" in sys.argv)
