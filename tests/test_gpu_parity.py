"""GPU parity tests (run with -m gpu on the B200 box): the CUDA hot path, called through the C ABI
(libcrgpu.so via ctypes), against the reference's golden outputs and the CPU oracle.

Tolerances.  Integer/index results (instance, polygon, RNG stream position) must be EXACT.  fp32
quantities that involve only + - * / sqrt must be BIT-EXACT.  Quantities behind a libm call
(sinf/cosf/powf/atan2f/acosf/asinf: the device evaluates them in fp64 and rounds once, glibc's fp32
routines are not always correctly rounded) may differ in the last ulp: 2e-6 relative on single values,
and the north-star bound RMSE <= 1e-4 on whole framebuffers (observed: 1e-9 .. 1e-5).
"""
import os

import numpy as np
import pytest

import crgpu
import oracle_lib as O
import reference_golden as RG
from conftest import GOLDEN, GOLDEN_SCENES, GOLDEN_FLAT, NO_BUNDLED

pytestmark = pytest.mark.gpu
RMSE_BOUND = 1e-4   # BASELINE.json north_star


def rmse(a, b):
    return float(np.sqrt(((a.astype(np.float64) - b.astype(np.float64)) ** 2).mean()))


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


@pytest.mark.parametrize("name", GOLDEN_FLAT)
def test_known_answer_records(name):
    h = np.fromfile(os.path.join(GOLDEN, name + ".hits.bin"), dtype=O.HIT_KAT_DTYPE)
    g = crgpu.GpuScene(os.path.join(GOLDEN, name + ".crscene"))
    xyp = np.stack([h["x"], h["y"], np.arange(len(h)) % g.samples], 1).astype(np.int32)
    k = np.frombuffer(g.trace_kat(xyp).tobytes(), dtype=O.HIT_KAT_DTYPE)
    for f in ("x", "y", "pixIdx", "instIndex", "polyIndex"):
        assert np.array_equal(k[f], h[f]), f
    # camera rays: bit-exact unless the thin lens is on (cosf/sinf of the lens angle)
    exact_rays = np.all(bits(k["o"]) == bits(h["o"]), axis=1) & np.all(bits(k["d"]) == bits(h["d"]), axis=1)
    np.testing.assert_allclose(k["o"], h["o"], rtol=2e-6, atol=1e-7)
    np.testing.assert_allclose(k["d"], h["d"], rtol=2e-6, atol=1e-7)
    assert exact_rays.mean() > 0.9
    # geometry of the hit is pure + - * / sqrt: bit-exact whenever the ray is
    hit = exact_rays & (h["instIndex"] >= 0)
    for f in ("distance", "hitPoint", "normal", "emission"):
        assert np.array_equal(bits(k[f][hit]), bits(h[f][hit])), f
    np.testing.assert_allclose(k["uv"], h["uv"], rtol=1e-5, atol=2e-6)
    np.testing.assert_allclose(k["out"], h["out"], rtol=1e-5, atol=2e-6)
    np.testing.assert_allclose(k["color"], h["color"], rtol=1e-5, atol=2e-6)
    # the RNG stream position after camera + bsdf sample must agree exactly (same number of draws, same branches)
    assert np.array_equal(bits(k["nextDraw"][exact_rays]), bits(h["nextDraw"][exact_rays]))
    g.close()


@pytest.mark.parametrize("name", GOLDEN_FLAT)
def test_framebuffer_vs_reference_golden(name):
    g = crgpu.GpuScene(os.path.join(GOLDEN, name + ".crscene"))
    ref = np.fromfile(os.path.join(GOLDEN, name + ".f32"), dtype=np.float32).reshape(g.H, g.W, 3)
    st = g.render_frame()
    img = g.read()
    assert st["paths"] == g.W * g.H * g.samples
    assert np.isfinite(img).all()
    assert rmse(img, ref) <= RMSE_BOUND, rmse(img, ref)
    g.close()


@pytest.mark.parametrize("name", ["g_legacy", "g_nodes"])
def test_tiling_batching_and_pass_splits_do_not_change_pixels(name):
    """The framebuffer must not depend on tile size, paths-in-flight budget or how passes are split
    (the reference is invariant to tile size and thread count, SURVEY App. C)."""
    path = os.path.join(GOLDEN, name + ".crscene")
    g = crgpu.GpuScene(path)
    g.render_frame()
    whole = g.read()
    # 16x16 tiles (reference tile grid, edge tiles ragged), tiny path budget -> one pass per batch
    g.clear()
    g.set_max_paths(1024)
    g.render_frame(tile=(16, 16))
    assert np.array_equal(bits(g.read()), bits(whole))
    # split passes 0..2 / 3..spp-1, odd tile size
    g.clear()
    g.set_max_paths(1 << 20)
    for y0 in range(0, g.H, 13):
        for x0 in range(0, g.W, 29):
            r = (x0, y0, min(x0 + 29, g.W), min(y0 + 13, g.H))
            g.render_tile(*r, pass_begin=0, pass_count=3)
            g.render_tile(*r, pass_begin=3, pass_count=g.samples - 3)
    assert np.array_equal(bits(g.read()), bits(whole))
    # resume from a host copy of the running average (renderer.c:283 reads renderBuffer back)
    g.clear()
    g.render_tile(0, 0, g.W, g.H, 0, 5)
    half = g.read()
    g.clear()
    g.write(half)
    g.render_tile(0, 0, g.W, g.H, 5, g.samples - 5)
    assert np.array_equal(bits(g.read()), bits(whole))
    g.close()


BUNDLED = [("hdr", 240, 135, 16, 32), ("scene", 320, 200, 16, 4), ("refraction", 240, 135, 8, 512), ("venus", 100, 160, 16, 25)]
# the other five bundled scenes: alpha nodes, textured fence, emissive + metal spheres, three large statues, uv-mapped sphere
BUNDLED += [(n, 96, 60, 8, 0) for n in ("alphanode", "fence", "glowmetal", "statues", "uvsphere")]


@pytest.mark.parametrize("name,W,H,spp,b", BUNDLED)
def test_bundled_scenes_vs_reference_framebuffer(name, W, H, spp, b, bundled_scene):
    """input/*.json scenes vs the framebuffers of the strict reference: the oracle, run here on the host cores, renders them bit
    for bit (it must reproduce the stored digest of the reference's frame), and the GPU frame is held to the RMSE bound."""
    scene = bundled_scene(name)
    if scene is None:
        pytest.skip(NO_BUNDLED)
    g = crgpu.GpuScene(scene, W, H, spp, b)
    st = g.render_frame(flags=crgpu.FLAG_COUNT)
    img = g.read()
    o = O.OracleScene(scene, W, H, spp, b)
    ref, c = o.render(threads=os.cpu_count(), count=True)
    assert RG.frame_digest(ref) == RG.golden()["frames"][RG.frame_key(name, W, H, spp, b)], "the oracle no longer renders the reference's frame"
    assert rmse(img, ref) <= RMSE_BOUND, rmse(img, ref)
    # identical paths => (almost) identical work counters; a last-ulp libm difference may re-route a few paths.
    # Rays with an exactly-zero direction component make the reference wander through up to ~1e5 BVH nodes
    # (NaN slab tests, see cr_node_test); the GPU culls them exactly, so its P and T may only be LOWER there.
    # The device slab test is the fused (fmaf) variant of bvh.c:318-324, the oracle the two-rounding one: rays that START on a
    # bounding-box face (every ray leaving an axis-aligned wall) get tMax = 0 +- 1 ulp, so which empty boxes are entered differs
    # in ~0.2% of the visits; hits do not (exact hit records are asserted in test_known_answer_records).
    assert abs(st["rays"] - c["rays"]) <= max(64, 2e-3 * c["rays"]), (st["rays"], c["rays"])
    # (fence.json — large axis-aligned planes — is where the fused/unfused difference shows most: 2.3% fewer mesh-instance visits
    # on the device, measured on the B200; the image and every hit record agree, so the counters are held to a one-sided band)
    for kg, kc in (("sphere_tests", "sphere_tests"), ("inst_visits", "inst_visits"), ("node_pairs", "node_pairs"), ("tri_tests", "tri_tests")):
        assert st[kg] <= c[kc] + max(64, 1e-2 * c[kc]) and st[kg] >= 0.9 * c[kc], (kg, st[kg], c[kc])
    assert st["paths"] == c["paths"]
    g.close()
    o.close()


FULL_SIZE = [   # BASELINE.json configs[1..4] geometry at reduced spp (the CPU cannot render the full jobs in a test)
    ("hdr", 1920, 1080, 4, 32, (500, 540)),          # C2
    ("refraction", 1920, 1080, 2, 512, (520, 540)),  # C3: 512-bounce glass paths; seeds wrap in 32 bits at 2500 spp (sampler KAT)
    ("venus", 2560, 1600, 2, 25, (800, 816)),        # C4: BVH-bound
    ("hdr", 7680, 4320, 1, 32, (2000, 2004)),        # C5 frame (8 GPUs in the bench; one GPU holds it fine)
]


@pytest.mark.parametrize("name,W,H,spp,b,band", FULL_SIZE)
def test_full_size_invariants(name, W, H, spp, b, band, bundled_scene):
    """Full-size frames: properties that do not need the CPU to render the frame — determinism, invariance to the tile
    decomposition and to the paths-in-flight budget, ray-count bounds, finite radiance — plus one band of
    rows checked against the oracle on the host cores (same seeds: they depend only on pixel, pass, spp, width)."""
    scene = bundled_scene(name)
    if scene is None:
        pytest.skip(NO_BUNDLED)
    import shard
    g = crgpu.GpuScene(scene, W, H, spp, b)
    st1 = g.render_tiles(shard.rank_rects(W, H, 64, 0, 1))
    a = g.read()
    g.clear()
    g.set_max_paths(4 << 20)
    st2 = None
    for rank in range(2):                                   # two "ranks" worth of 128x128 tiles, small batches
        s_ = g.render_tiles(shard.rank_rects(W, H, 128, rank, 2))
        st2 = s_ if st2 is None else {k: st2[k] + s_[k] for k in st2}
    bimg = g.read()
    assert np.array_equal(bits(a), bits(bimg))
    assert st1["rays"] == st2["rays"] and st1["paths"] == W * H * spp
    assert st1["paths"] <= st1["rays"] <= b * st1["paths"]
    assert np.isfinite(a).all()     # (negative values are legitimate: texture.c:66-79 extrapolates when x*W-0.5 < 0)
    o = O.OracleScene(scene, W, H, spp, b)
    ref = np.zeros((H, W, 3), np.float32)
    o.render(threads=os.cpu_count(), tile=(0, band[0], W, band[1]), rgb=ref)
    rows = slice(H - band[1], H - band[0])
    assert rmse(a[rows], ref[rows]) <= RMSE_BOUND
    g.close()
    o.close()


def test_srgb8_output_byte_exact():
    """colorToSRGB + the (unsigned char) store (color.h:60-84, renderer.c:297-300): BYTE-exact against the oracle (glibc powf).
    The device evaluates powf in fp64 and rounds once; the two differ in the last ulp for ~0.06% of inputs but never across a
    byte boundary — checked here over the rendered frame AND exhaustively over EVERY float in [0.0031308, 1.5] (74.6 M values,
    the whole powf branch up to well past saturation), plus the linear branch, negatives, inf and NaN."""
    g = crgpu.GpuScene(os.path.join(GOLDEN, "g_nodes.crscene"))
    g.render_frame()
    img = g.read()
    out8 = g.srgb8()
    exp = np.zeros_like(out8)
    O.lib().cro_to_srgb8(img.ctypes.data, exp.ctypes.data, img.shape[0] * img.shape[1])
    assert np.array_equal(out8, exp)
    g.close()
    lo, hi = np.array([0.0031308, 1.5], dtype=np.float32).view(np.uint32)
    W, H = 4096, 6080                                      # 74.7 M floats
    n = W * H * 3
    assert n >= int(hi) - int(lo) + 1 + 4096
    vals = np.zeros(n, dtype=np.uint32)
    k = int(hi) - int(lo) + 1
    vals[:k] = np.arange(int(lo), int(hi) + 1, dtype=np.uint32)
    rng = np.random.default_rng(5)
    extra = rng.integers(0, 2 ** 32, size=n - k - 8, dtype=np.uint64).astype(np.uint32)          # arbitrary bit patterns: negatives, NaNs, denormals
    vals[k:k + len(extra)] = extra
    vals[-8:] = np.array([0.0, -0.0, np.inf, -np.inf, np.nan, 1.0, 0.0031308, -1e-3], dtype=np.float32).view(np.uint32)
    g = crgpu.GpuScene(os.path.join(GOLDEN, "g_single.crscene"), W, H, 1, 1)
    fb = vals.view(np.float32).reshape(H, W, 3)
    g.write(fb)
    out8 = g.srgb8()
    exp = np.zeros_like(out8)
    O.lib().cro_to_srgb8(fb.ctypes.data, exp.ctypes.data, W * H)
    bad = np.nonzero(out8.ravel() != exp.ravel())[0]
    assert len(bad) == 0, (len(bad), vals[bad[:8]], out8.ravel()[bad[:8]], exp.ravel()[bad[:8]])
    g.close()


def test_zero_bounces_is_black():
    """prefs.bounces == 0 (accepted by the reference and by the loader): every sample is black; the L buffer is write-once
    in the kernels, so the driver has to clear it when no bounce runs (crgpu_api.cu render_pixels)."""
    g = crgpu.GpuScene(os.path.join(GOLDEN, "g_single.crscene"), force_bounces=0)
    g.write(np.full((g.H, g.W, 3), 7.0, dtype=np.float32))     # poison: the running average must overwrite it with zeros
    g.clear()
    st = g.render_frame()
    assert st["rays"] == 0 and st["paths"] == g.W * g.H * g.samples
    img = g.read()
    assert not img.any()
    g.close()


def test_argument_errors_are_reported():
    g = crgpu.GpuScene(os.path.join(GOLDEN, "g_single.crscene"))
    with pytest.raises(crgpu.CrgpuError):
        g.render_tile(0, 0, g.W + 1, g.H)
    with pytest.raises(crgpu.CrgpuError):
        g.render_tile(5, 5, 5, 9)
    with pytest.raises(crgpu.CrgpuError):
        g.render_tile(0, 0, g.W, g.H, pass_begin=g.samples, pass_count=1)
    with pytest.raises(crgpu.CrgpuError):
        crgpu.GpuScene(os.path.join(GOLDEN, "g_single.crscene"), device=99)
    g.close()


def test_empty_pass_range_is_a_no_op():
    g = crgpu.GpuScene(os.path.join(GOLDEN, "g_single.crscene"))
    st = g.render_tile(0, 0, g.W, g.H, 0, 0)
    assert st["rays"] == 0 and not g.read().any()
    g.close()


def test_render_tiles_union_equals_whole_frame():
    """crgpu_render_tiles: a rank's share of the tile grid as ONE wavefront (the multi-GPU bench path)."""
    import shard
    g = crgpu.GpuScene(os.path.join(GOLDEN, "g_legacy.crscene"))
    g.render_frame()
    whole = g.read()
    g.clear()
    for rank in range(3):
        st = g.render_tiles(shard.rank_rects(g.W, g.H, 16, rank, 3))
        assert st["paths"] > 0
    assert np.array_equal(bits(g.read()), bits(whole))
    with pytest.raises(crgpu.CrgpuError):
        g.render_tiles([(0, 0, g.W + 5, 4)])
    g.close()


def test_seed_wraps_in_32_bits_on_the_device(bundled_scene):
    """sampler.c:42: seed = hash64(u32(pixIdx) * u32(maxPasses) + u32(pass)) — the product wraps for C3 (2.07 M pixels x 2500 spp)
    and C5 (33 M pixels x 4000 spp).  Camera rays (no lens in refraction.json: pure + - * / sqrt of two draws) must be bit-exact
    against the oracle for pixels/passes beyond the wrap, and a tile rendered for the LAST passes must match the oracle."""
    scene = bundled_scene("refraction")
    if scene is None:
        pytest.skip(NO_BUNDLED)
    W, H, spp, b = 1920, 1080, 2500, 512
    g = crgpu.GpuScene(scene, W, H, spp, b)
    o = O.OracleScene(scene, W, H, spp, b)
    xyp = np.array([[5, 900, 2499], [1919, 1079, 2499], [960, 1000, 1234], [0, 895, 17], [100, 10, 2499]], dtype=np.int32)
    assert ((xyp[:4, 1].astype(np.int64) * W + xyp[:4, 0]) * spp + xyp[:4, 2] >= 2 ** 32).all()      # wrapped seeds
    k = np.frombuffer(g.trace_kat(xyp).tobytes(), dtype=O.HIT_KAT_DTYPE)
    for i, (x, y, p) in enumerate(xyp):
        ref = o.trace_kat(int(x), int(y), int(p))
        assert np.array_equal(bits(k["d"][i]), bits(ref["d"])) and np.array_equal(bits(k["o"][i]), bits(ref["o"])), (x, y, p)
        assert k["instIndex"][i] == ref["instIndex"] and np.array_equal(bits(k["distance"][i:i + 1]), bits(np.array([ref["distance"]], np.float32)))
    tile, passes = (128, 1000, 192, 1064), (2490, 10)
    g.render_tile(*tile, pass_begin=passes[0], pass_count=passes[1])
    img = g.read()
    ref = np.zeros((H, W, 3), np.float32)
    o.render(threads=os.cpu_count(), tile=tile, passes=passes, rgb=ref)
    rows, cols = slice(H - tile[3], H - tile[1]), slice(tile[0], tile[2])
    scale = spp / passes[1]           # the running average started from zero at pass 2490: rescale to "mean of these 10 samples"
    assert np.isfinite(img[rows, cols]).all()
    # RMSE <= 1e-4 is the bound for the full 2500-sample mean; a 10-sample mean of the same per-sample errors is sqrt(250) x noisier
    assert rmse(img[rows, cols] * scale, ref[rows, cols] * scale) <= RMSE_BOUND * np.sqrt(scale)
    assert (bits(img[rows, cols]) == bits(ref[rows, cols])).all(axis=2).mean() > 0.5
    g.close()
    o.close()


def test_c5_tile_at_full_sample_count(bundled_scene):
    """BASELINE C5 geometry (hdr.json 7680x4320, 4000 spp): one 64x64 tile at the top of the frame for ALL 4000 passes against
    the oracle (16 M samples; seeds wrap: 33 M pixels x 4000)."""
    scene = bundled_scene("hdr")
    if scene is None:
        pytest.skip(NO_BUNDLED)
    W, H, spp, b = 7680, 4320, 4000, 32
    tile = (3840, 4200, 3904, 4264)
    g = crgpu.GpuScene(scene, W, H, spp, b)
    g.render_tile(*tile)
    img = g.read()
    g.close()
    o = O.OracleScene(scene, W, H, spp, b)
    ref = np.zeros((H, W, 3), np.float32)
    o.render(threads=os.cpu_count(), tile=tile, rgb=ref)
    o.close()
    rows, cols = slice(H - tile[3], H - tile[1]), slice(tile[0], tile[2])
    assert np.isfinite(img[rows, cols]).all()
    assert rmse(img[rows, cols], ref[rows, cols]) <= RMSE_BOUND


def test_prepared_scene_is_reusable_and_the_device_cache_is_transparent():
    """crgpu_prepare once, crgpu_scene_create_prepared many times (what renderFrame does per frame): every replica renders the same
    bits as a scene made by crgpu_scene_create, also after create/destroy cycles that recycle device blocks from the cache."""
    import crhost
    path = os.path.join(GOLDEN, "g_nodes.crscene")
    g = crgpu.GpuScene(path)
    g.render_frame()
    whole = g.read()
    g.close()
    R = crhost.Renderer(path, gpus=1, tile=16)
    R.prepare()
    for _ in range(3):
        h = crgpu.GpuScene(None, samples=R.samples, bounces=R.bounces, prepared=R.prepared())
        h.render_frame()
        assert np.array_equal(bits(h.read()), bits(whole))
        h.close()
    for _ in range(2):                       # renderFrame in C: upload -> tiles -> read back
        secs, rays = R.render()
        assert rays > 0 and np.array_equal(bits(R.framebuffer()), bits(whole))
    R.close()
    assert crgpu.lib().crgpu_device_trim(0) == 0
    g = crgpu.GpuScene(path)
    g.render_frame()
    assert np.array_equal(bits(g.read()), bits(whole))
    g.close()


def _decode_png(path):
    import struct, zlib
    b = open(path, "rb").read()
    pos, idat, W, H = 8, b"", 0, 0
    while pos < len(b):
        n, tag = struct.unpack(">I4s", b[pos:pos + 8])
        data = b[pos + 8:pos + 8 + n]
        if tag == b"IHDR":
            W, H = struct.unpack(">II", data[:8])
        elif tag == b"IDAT":
            idat += data
        pos += 12 + n
    raw = np.frombuffer(zlib.decompress(idat), dtype=np.uint8).reshape(H, W * 3 + 1)
    return raw[:, 1:].reshape(H, W, 3)


def _run_cli(args, tmp_path):
    import subprocess
    from conftest import ROOT
    exe = os.path.join(ROOT, "c-ray_b200", "cray_b200")
    r = subprocess.run([exe] + args, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-2000:]
    return r.stdout


def test_host_c_renderer_cli(tmp_path):
    """The host C mirror (renderFrame + gpuRenderThread + tile queue + PNG writer) end to end."""
    scene = os.path.join(GOLDEN, "g_legacy.crscene")
    f32, png = str(tmp_path / "o.f32"), str(tmp_path / "o.png")
    out = _run_cli([scene, "-t", "16x16", "-o", png, "--dump-f32", f32], tmp_path)
    assert "Finished render" in out
    g = crgpu.GpuScene(scene)
    g.render_frame()
    assert np.array_equal(bits(np.fromfile(f32, dtype=np.float32)), bits(g.read().ravel()))
    assert np.array_equal(_decode_png(png), g.srgb8())
    g.close()


@pytest.mark.parametrize("gpus", [2, 4, 8])
def test_host_c_renderer_multi_gpu_nccl_gather(tmp_path, gpus, bundled_scene):
    """-j N: N gpuRenderThreads share the tile queue, tiles are gathered on device 0 by libcrgpu_nccl.so; bit-identical to -j 1.
    (Round 1 saw one wrong tile at -j 8: the tile set's pixel list was uploaded with a legacy-stream cudaMemcpy that the first
    k_generate on the scene's non-blocking stream could overtake; crgpu_render_tiles now uploads on the scene's stream.)"""
    if crgpu.device_count() < gpus:
        pytest.skip(f"needs {gpus} GPUs")
    scene = bundled_scene("hdr")
    args = [scene, "-d", "480x270", "-s", "64", "-t", "32x32"] if scene else [os.path.join(GOLDEN, "g_nodes.crscene"), "-t", "16x16"]
    a, b = str(tmp_path / "a.f32"), str(tmp_path / "b.f32")
    _run_cli(args + ["-j", "1", "--dump-f32", a, "-q"], tmp_path)
    _run_cli(args + ["-j", str(gpus), "--dump-f32", b, "-q"], tmp_path)
    assert np.array_equal(bits(np.fromfile(a, dtype=np.float32)), bits(np.fromfile(b, dtype=np.float32)))


def _bench(args, nproc=1, timeout=900):
    import json
    import subprocess
    import sys
    from conftest import ROOT
    from test_multi_rank import free_port
    cmd = [sys.executable]
    if nproc > 1:
        cmd += ["-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(nproc), "--master-addr", "127.0.0.1", "--master-port", str(free_port())]
    cmd += [os.path.join(ROOT, "bench.py"), "--gpus", str(nproc)] + args
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=timeout, cwd=ROOT)
    assert r.returncode == 0, (r.stdout + r.stderr)[-3000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, r.stdout[-2000:]
    return json.loads(lines[0])


def test_bench_line_contract_small_workload(tmp_path):
    """bench.py end to end on the C1 geometry (input/scene.json 320x200x16spp): the JSON line carries every key of the contract, the
    frame coming back through libcrhost's renderFrame is the one the resident path rendered, it is finite, and --dump-outputs
    writes that frame."""
    import zlib
    line = _bench(["--workload", "scene", "--steps", "2", "--warmup", "1", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)])
    fb = np.load(tmp_path / "framebuffer.npy")
    assert fb.shape == (200, 320, 3) and fb.dtype == np.float32 and f"{zlib.crc32(fb.tobytes()):08x}" == line["value_path_crc32"]
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "dtype", "config", "e2e",
              "gpu_launches", "clocks", "roofline", "frame_crc32"):
        assert k in line, k
    assert line["value"] > 0 and line["e2e"]["value"] > 0 and line["gpu_launches"] > 0
    assert line["frame_crc32"] == line["value_path_crc32"] and line["frame_finite"]
    assert line["e2e"]["h2d_bytes_per_step"] > 1000 and line["roofline"]["frac"] is not None


@pytest.mark.parametrize("ranks", [2, 4, 8])
def test_torchrun_ranks_render_the_single_gpu_frame(ranks):
    """The measured multi-GPU path: one process per GPU (torchrun), tiles dealt out by the C dispatcher, ONE NCCL gather in C.
    The frame on rank 0 must have the CRC of the 1-GPU frame."""
    if crgpu.device_count() < ranks:
        pytest.skip(f"needs {ranks} GPUs")
    common = ["--workload", "hdr", "--width", "480", "--height", "270", "--spp", "64", "--steps", "1", "--warmup", "1", "--no-cpu-baseline"]
    one = _bench(common, 1)
    many = _bench(common, ranks)
    assert many["n_gpus"] == ranks and many["frame_crc32"] == one["frame_crc32"] == many["value_path_crc32"]
    assert abs(many["rays_per_sample"] - one["rays_per_sample"]) < 1e-9
