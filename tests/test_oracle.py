"""CPU tests: the oracle (oracle/cray_oracle.c) against the reference's own outputs.

The golden files were produced by the unmodified reference built with -ffp-contract=off
(tests/golden/make_golden.py).  The bar for the oracle is BIT-EXACT fp32.
"""
import os

import numpy as np
import pytest

import oracle_lib as O
import reference_golden as RG
from conftest import GOLDEN, GOLDEN_SCENES, GOLDEN_FLAT, NO_BUNDLED


def test_sampler_kat_bit_exact():
    k = np.fromfile(os.path.join(GOLDEN, "kat.bin"), dtype=np.uint32).reshape(-1, 16)
    assert len(k) == 10
    for row in k:
        pix, p, mp = (int(v) for v in row[:3])
        mine = O.sampler_kat(pix, p, mp, 13)
        assert np.array_equal(row[3:], mine.view(np.uint32)), (pix, p, mp)


def test_sampler_seed_wraps_in_32_bits():
    # sampler.c:42: pixelIndex * maxPasses + pass is uint32 arithmetic
    a = O.sampler_kat(2073599, 2499, 2500, 4)
    wrapped = (2073599 * 2500 + 2499) & 0xFFFFFFFF
    b = O.sampler_kat(wrapped, 0, 1, 4)
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))


def test_draw_range_inclusive_one():
    # random.c:17: 2^-32 * (float)u32 rounds up to exactly 1.0f for u32 >= 2^32-128
    v = O.sampler_kat(0, 0, 1, 4096)
    assert v.min() >= 0.0 and v.max() <= 1.0


@pytest.mark.parametrize("name", GOLDEN_FLAT)
def test_framebuffer_bit_exact(name):
    sc = O.OracleScene(os.path.join(GOLDEN, name + ".crscene"))
    ref = np.fromfile(os.path.join(GOLDEN, name + ".f32"), dtype=np.float32).reshape(sc.H, sc.W, 3)
    img = sc.render(threads=4)
    assert np.array_equal(img.view(np.uint32), ref.view(np.uint32))
    sc.close()


@pytest.mark.parametrize("name", GOLDEN_FLAT)
def test_hit_records_bit_exact(name):
    sc = O.OracleScene(os.path.join(GOLDEN, name + ".crscene"))
    h = np.fromfile(os.path.join(GOLDEN, name + ".hits.bin"), dtype=O.HIT_KAT_DTYPE)
    assert len(h) == 96
    for i, r in enumerate(h):
        m = sc.trace_kat(int(r["x"]), int(r["y"]), i % sc.s.prefs.sample_count)
        assert r.tobytes() == m.tobytes(), (name, i)
    sc.close()


@pytest.mark.parametrize("name", GOLDEN_FLAT)
def test_tiles_and_pass_ranges_compose(name):
    """Tile size, thread count and splitting the passes never change a pixel (renderer.c:271-320)."""
    sc = O.OracleScene(os.path.join(GOLDEN, name + ".crscene"))
    ref = np.fromfile(os.path.join(GOLDEN, name + ".f32"), dtype=np.float32).reshape(sc.H, sc.W, 3)
    img = np.zeros_like(ref)
    spp = sc.s.prefs.sample_count
    for (pb, pc) in ((0, 3), (3, spp - 3)):
        for y0 in range(0, sc.H, 16):
            for x0 in range(0, sc.W, 16):
                sc.render(threads=1, tile=(x0, y0, min(x0 + 16, sc.W), min(y0 + 16, sc.H)), passes=(pb, pc), rgb=img)
    assert np.array_equal(img.view(np.uint32), ref.view(np.uint32))
    sc.close()


def test_counters_consistent():
    sc = O.OracleScene(os.path.join(GOLDEN, "g_legacy.crscene"))
    _, c = sc.render(threads=2, count=True)
    assert c["paths"] == sc.W * sc.H * sc.s.prefs.sample_count
    assert c["paths"] <= c["rays"] <= c["paths"] * sc.s.prefs.bounces
    assert c["max_depth"] <= sc.s.prefs.bounces and c["max_stack"] <= 64
    assert c["node_pairs"] > 0 and c["tri_tests"] > 0 and c["sphere_tests"] > 0 and c["inst_visits"] > 0
    sc.close()


def test_srgb8_matches_reference_formula():
    rgb = np.array([0.0, 0.001, 0.0031308, 0.2, 0.5, 1.0, 1.5, 7.0, 0.99999], dtype=np.float32)
    rgb = np.resize(rgb, 9).astype(np.float32)
    out = np.zeros(9, dtype=np.uint8)
    O.lib().cro_to_srgb8(rgb.ctypes.data, out.ctypes.data, 3)
    exp = []
    for c in rgb:
        s = 12.92 * c if c <= 0.0031308 else 1.055 * c ** 0.4166666667 - 0.055
        exp.append(min(int(min(s * 255.0, 255.0)), 255))
    assert np.abs(out.astype(int) - np.array(exp)).max() <= 1


@pytest.mark.parametrize("name,W,H,spp,b", [("hdr", 96, 54, 4, 32), ("scene", 80, 50, 4, 4), ("refraction", 64, 36, 2, 512), ("venus", 40, 64, 4, 25),
                                            ("alphanode", 96, 60, 8, 0), ("fence", 96, 60, 8, 0), ("glowmetal", 96, 60, 8, 0),
                                            ("statues", 96, 60, 8, 0), ("uvsphere", 96, 60, 8, 0)])
def test_bundled_scenes_against_reference_framebuffers(name, W, H, spp, b, bundled_scene):
    """Bundled input/*.json scenes: the oracle vs the framebuffers the strict reference rendered (their digests,
    tests/golden/reference.json): bit-exact."""
    scene = bundled_scene(name)
    if scene is None:
        pytest.skip(NO_BUNDLED)
    sc = O.OracleScene(scene, W, H, spp, b)
    img = sc.render(threads=os.cpu_count())
    assert RG.frame_digest(img) == RG.golden()["frames"][RG.frame_key(name, W, H, spp, b)]
    sc.close()


@pytest.mark.parametrize("name,W,H,spp,b", [("hdr", 1920, 1080, 2, 32), ("venus", 2560, 1600, 1, 25), ("refraction", 1920, 1080, 1, 512)])
def test_full_size_frames_bit_exact_against_live_reference(name, W, H, spp, b, bundled_scene):
    """BASELINE.json configs C2 / C4 / C3 at their full image sizes (few spp): the strict reference build (the digest of its
    frame, tests/golden/reference.json) and the oracle produce the same fp32 frame bit for bit.  (The GPU suite then checks
    bands of these frames against the oracle.)"""
    scene = bundled_scene(name)
    if scene is None:
        pytest.skip(NO_BUNDLED)
    sc = O.OracleScene(scene, W, H, spp, b)
    img = sc.render(threads=os.cpu_count())
    assert RG.frame_digest(img) == RG.golden()["frames"][RG.frame_key(name, W, H, spp, b)]
    sc.close()


def test_glass_total_internal_reflection_with_draw_of_exactly_one(bundled_scene):
    """glass.c:47 declares `refracted` uninitialised and reads it when refract() failed (total internal reflection) AND the
    reflect/refract draw is exactly 1.0f (129 of 2^32 draws): the compiled reference scatters along (0, 0, <stale stack word>).
    Known occurrence (round-1 judge): hdr.json 1920x1080x1000spp, pixel x=165 y(up)=768, pass 576, bounce 2.  The oracle and the
    device DEFINE that case as a reflection (DESIGN.md deviation #3), so (a) the sample is finite, (b) the pixel differs from the
    strict reference by at most that one sample's share, (c) every pixel around it stays bit-identical to the reference."""
    scene = bundled_scene("hdr")
    if scene is None:
        pytest.skip(NO_BUNDLED)
    W, H, spp, b = 1920, 1080, 1000, 32
    sc = O.OracleScene(scene, W, H, spp, b)
    one = np.zeros((H, W, 3), np.float32)
    sc.render(threads=1, tile=(165, 768, 166, 769), passes=(576, 1), rgb=one)       # running average from zero: (0*575 + L)/576
    sample = one[H - 1 - 768, 165].astype(np.float64) * 577.0
    assert np.isfinite(sample).all(), sample
    img = np.zeros((H, W, 3), np.float32)
    sc.render(threads=os.cpu_count(), tile=RG.TIR_BLOCK, rgb=img)
    blk = img[H - 772:H - 764, 160:172]
    assert np.isfinite(blk).all()
    with np.load(RG.FULL_SAMPLES) as z:          # the block of the strict reference's full frame
        ref = z["tir_block"]
    same = (blk.view(np.uint32) == ref.view(np.uint32)).all(axis=2)
    assert same.sum() == same.size - 1 and not same[772 - 1 - 768, 165 - 160], same
    # one of 1000 samples took another direction after its third hit: bounded by that sample's own radiance / spp
    assert np.abs(blk[772 - 1 - 768, 5].astype(np.float64) - ref[772 - 1 - 768, 5]).max() <= (np.abs(sample).max() + 64.0) / spp
    sc.close()


def test_zero_bounces_is_black():
    """prefs.bounces == 0: pathTrace's loop never runs (pathtrace.c:36-59) — the reference renders an all-zero frame
    (checked against cray_ref_strict with "bounces": 0 in the JSON)."""
    sc = O.OracleScene(os.path.join(GOLDEN, "g_single.crscene"))
    sc.s.prefs.bounces = 0
    img = sc.render(threads=2)
    assert not img.any()
    sc.close()
