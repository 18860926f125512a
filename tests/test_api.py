"""c-ray's public library API (reference src/c-ray.h) served by libcrhost.so (include/cray_api.h, c-ray_b200/host/cr_api.c).

CPU: every declared entry point is exported; argument parsing, option tags, scene loading through crLoadSceneFromBuf and
the pref getters behave like reference src/utils/args.c / src/c-ray.c; without a GPU crStartRenderer fails loudly.
GPU: the reference's OWN main program (src/main.c compiled in place by oracle/Makefile against this library,
oracle/_ref/cray_main_b200) renders a bundled scene and writes the PNG the python path produces.
"""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

from conftest import ROOT, GOLDEN

MAIN = os.path.join(ROOT, "oracle", "_ref", "cray_main_b200")
REF_DIR = os.path.join(ROOT, "oracle", "_ref")


def declared():
    text = open(os.path.join(ROOT, "include", "cray_api.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(cr[A-Z]\w+|isDebug)\s*\(", text)))


def test_api_exports_every_declared_entry_point():
    L = C.CDLL(os.path.join(ROOT, "c-ray_b200", "libcrhost.so"))
    names = declared()
    assert len(names) >= 50 and "crLoadSceneFromBuf" in names and "crStartRenderer" in names
    for n in names:
        getattr(L, n)


API_SCRIPT = r"""
import ctypes as C, os, sys
L = C.CDLL(os.path.join(sys.argv[1], "c-ray_b200", "libcrhost.so"))
L.crPathArg.restype = C.c_char_p; L.crGetAssetPath.restype = C.c_char_p
L.crGetOutputPath.restype = C.c_char_p; L.crGetFileName.restype = C.c_char_p
L.crOptionIsSet.argtypes = [C.c_char_p]; L.crOptionIsSet.restype = C.c_bool
L.crLoadSceneFromBuf.argtypes = [C.c_char_p]
args = [b"c-ray", b"g_legacy", b"-d", b"40x24", b"-s", b"3", b"-t", b"8x8", b"-j", b"1", b"--gpu"]
argv = (C.c_char_p * (len(args) + 1))(*args, None)
L.crInitialize()
L.crParseArgs(len(args), argv)
assert L.crPathArg() == b"g_legacy.json", L.crPathArg()            # <arg>.json fallback (args.c:82-88)
assert L.crOptionIsSet(b"inputFile") and L.crOptionIsSet(b"-gpu") and L.crOptionIsSet(b"dims_override") and not L.crOptionIsSet(b"nope")
L.crInitRenderer()
assert L.crGetAssetPath() == b"./"
assert L.crLoadSceneFromBuf(open("g_legacy.json", "rb").read()) == 0
assert (L.crGetImageWidth(), L.crGetImageHeight(), L.crGetSampleCount(), L.crGetTileWidth(), L.crGetTileHeight(), L.crGetThreadCount()) == (40, 24, 3, 8, 8, 1)
assert L.crGetBounces() == 6 and L.crGetOutputPath() == b"output/" and L.crGetFileName() == b"g"
L.crSetSampleCount(5); L.crSetBounces(9); L.crSetImageWidth(64)
assert (L.crGetSampleCount(), L.crGetBounces(), L.crGetImageWidth()) == (5, 9, 64)
assert L.crLoadSceneFromBuf(b"{ not json") == -1
L.crStartRenderer()          # no GPU here: must complain, must not produce an image
L.crWriteImage()
L.crDestroyRenderer(); L.crDestroyOptions()
print("API-OK")
"""


def test_api_semantics_without_gpu(tmp_path):
    """Runs in a subprocess (the API keeps process-global state like the reference's g_renderer)."""
    import json
    bounces = json.load(open(os.path.join(GOLDEN, "g_legacy.json")))["renderer"]["bounces"]
    script = API_SCRIPT.replace("L.crGetBounces() == 6", f"L.crGetBounces() == {bounces}")
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run(["python", "-c", script, ROOT], cwd=GOLDEN, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=120, env=env)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "API-OK" in r.stdout
    assert "render failed" in r.stderr and "CUDA" in r.stderr       # fails loudly: there is no CPU rendering path
    assert not os.path.exists(os.path.join(GOLDEN, "g_0000.png"))


@pytest.mark.gpu
def test_reference_main_program_on_the_b200_path(tmp_path, monkeypatch):
    """reference src/main.c (unmodified, built by oracle/Makefile) + libcrhost.so: input/hdr.json -> PNG."""
    import crgpu
    from test_gpu_parity import _decode_png
    if not os.path.exists(MAIN):
        pytest.skip("oracle/_ref/cray_main_b200 is built where /root/reference exists and travels with the repo")
    r = subprocess.run([MAIN, "input/hdr.json", "-d", "96x54", "-s", "4", "-t", "32x32"], cwd=REF_DIR, stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0 and "Saving result in" in r.stdout, r.stdout[-2000:]
    path = re.search(r'Saving result in "([^"]+)"', r.stdout).group(1)
    png = _decode_png(os.path.join(REF_DIR, path))
    monkeypatch.chdir(REF_DIR)
    g = crgpu.GpuScene(os.path.join("input", "hdr.json"), 96, 54, 4)
    g.render_frame()
    assert np.array_equal(png, g.srgb8())
    g.close()
    os.remove(os.path.join(REF_DIR, path))


@pytest.mark.gpu
def test_reference_renderframe_with_the_gpu_worker_in_its_thread_slot(tmp_path, bundled_scene):
    """INTEGRATION.md §2, compiled and run: oracle/_ref/cray_ref_gpu is the UNMODIFIED reference (its loader, BVH builder, tile
    queue, renderFrame, stats loop) built by oracle/Makefile with the two integration files a maintainer adds
    (c-ray_b200/integration/gpu_thread.c + flatten_world.c) and libcrgpu.so.  With CRAY_GPU=1 renderFrame's thread-function slot
    (renderer.c:92-105) is filled with gpuRenderThread; the fp32 renderBuffer must match the CPU reference's."""
    import oracle_lib as O
    import reference_golden as RG
    exe = os.path.join(REF_DIR, "cray_ref_gpu")
    scene = bundled_scene("scene")
    if not (os.path.exists(exe) and scene):
        pytest.skip("oracle/_ref/cray_ref_gpu and oracle/_ref/input are built by build() where the reference sources are present")
    out = str(tmp_path / "gpu.f32")
    r = subprocess.run([exe, "render", "input/scene.json", "320", "200", "16", "4", "1", "0", "0", out], cwd=REF_DIR,
                       env=dict(os.environ, CRAY_GPU="1"), stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0 and "REF_RENDER" in r.stdout, r.stdout[-2000:]
    got = np.fromfile(out, dtype=np.float32)
    o = O.OracleScene(scene, 320, 200, 16, 4)
    ref = o.render(threads=os.cpu_count()).ravel()       # the strict reference's frame, bit for bit (checked by its digest)
    o.close()
    assert RG.frame_digest(ref) == RG.golden()["frames"][RG.frame_key("scene", 320, 200, 16, 4)]
    assert got.shape == ref.shape and np.isfinite(got).all()
    rmse = float(np.sqrt(((got.astype(np.float64) - ref) ** 2).mean()))
    assert rmse <= 1e-4, rmse
    # and the same binary WITHOUT the flag is still the CPU reference, bit for bit
    out2 = str(tmp_path / "cpu.f32")
    r = subprocess.run([exe, "render", "input/scene.json", "80", "50", "4", "4", "2", "0", "0", out2], cwd=REF_DIR,
                       env={k: v for k, v in os.environ.items() if k != "CRAY_GPU"}, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0
    assert RG.frame_digest(np.fromfile(out2, dtype=np.float32)) == RG.golden()["frames"][RG.frame_key("scene", 80, 50, 4, 4)]
