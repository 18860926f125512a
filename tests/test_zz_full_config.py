"""The headline parity numbers: per-pixel RMSE of the GPU frame against the UNMODIFIED reference (strict build, oracle/_ref/
cray_ref_strict) AT THE BASELINE CONFIGURATIONS — BASELINE.json configs[1..3]: hdr.json 1920x1080x1000spp/32 bounces (the
configuration the metric is quoted on, bound 1e-4 at matched PCG seeds), refraction.json 1920x1080x2500spp/512 bounces,
venus.json 2560x1600x1000spp.  The reference frames were rendered once (tests/reference_golden.py --full, 4.6 CPU-minutes to
~1 CPU-hour each on 8 cores) and a fixed sample of 4096 pixels of each is stored in tests/golden/full_config_samples.npz; the GPU
renders the whole frame and is compared at those pixels.  A configuration without a stored sample is skipped, never substituted.

What is compared, over the sampled pixels: (1) the set of non-finite pixels — the GPU frame may have none the reference does not
have; (2) RMSE and max |diff| over the pixels finite on both sides; (3) ray counts.  The numbers are printed and queued for the
pytest terminal summary BEFORE any assert, so a failing run still shows them.
Collected last (file name) so that a slow host never starves the other tests."""
import json
import time

import numpy as np
import pytest

import conftest
import reference_golden as RG
from conftest import NO_BUNDLED

FULL = [("hdr", 1920, 1080, 1000, 32), ("refraction", 1920, 1080, 64, 512), ("venus", 2560, 1600, 32, 25),
        ("refraction", 1920, 1080, 2500, 512), ("venus", 2560, 1600, 1000, 25)]


def rmse_bound(spp):
    """north_star: RMSE <= 1e-4 at the configurations' own sample counts (>= 1000 spp).  The only source of error is a path that
    takes another branch after a last-ulp libm difference (DESIGN.md deviation 1); such a sample moves its pixel by delta/spp, and
    with a fixed per-sample rate the frame RMSE goes as 1/sqrt(spp).  The reduced-spp frames of the same geometry are therefore held
    to 1e-4 * sqrt(1000/spp) — the same per-sample divergence rate the 1e-4 bound allows at 1000 spp (measured on B200: refraction
    64 spp 2.1e-4 vs bound 4.0e-4, venus 32 spp 1.3e-4 vs 5.6e-4, hdr 1000 spp 1.05e-5 vs 1e-4)."""
    return 1e-4 if spp >= 1000 else 1e-4 * (1000.0 / spp) ** 0.5


def compare_frames(gpu, ref):
    """dict of parity figures between two fp32 (H,W,3) frames; no asserts."""
    gbad = ~np.isfinite(gpu).all(axis=2)
    rbad = ~np.isfinite(ref).all(axis=2)
    ok = ~(gbad | rbad)
    d = gpu[ok].astype(np.float64) - ref[ok]
    ys, xs = np.nonzero(gbad & ~rbad)
    return {"rmse": float(np.sqrt(np.mean(d * d))) if d.size else float("nan"),
            "max_abs_diff": float(np.abs(d).max()) if d.size else float("nan"),
            "pixels": int(gpu.shape[0] * gpu.shape[1]), "pixels_compared": int(ok.sum()),
            "pixels_bit_identical": int((gpu.view(np.uint32) == ref.view(np.uint32)).all(axis=2).sum()),
            "nonfinite_gpu": int(gbad.sum()), "nonfinite_reference": int(rbad.sum()),
            "nonfinite_gpu_only": [[int(x), int(gpu.shape[0] - 1 - y)] for x, y in zip(xs[:8], ys[:8])]}


def record(out):
    conftest.SUMMARY_LINES.append("FULL-CONFIG-RMSE " + json.dumps(out))
    print(conftest.SUMMARY_LINES[-1])


@pytest.mark.gpu
@pytest.mark.parametrize("name,W,H,spp,b", FULL)
def test_full_config_rmse_vs_strict_reference(name, W, H, spp, b, bundled_scene):
    import crgpu
    key = RG.frame_key(name, W, H, spp, b)
    with np.load(RG.FULL_SAMPLES) as z:
        if key not in z.files:
            pytest.skip(f"no stored sample of the reference frame {key} (rendering it takes about a CPU-hour)")
        ref = z[key][None]
    scene = bundled_scene(name)
    if scene is None:
        pytest.skip(NO_BUNDLED)
    t0 = time.time()
    g = crgpu.GpuScene(scene, W, H, spp, b)
    st = g.render_frame()
    gpu = g.read().reshape(-1, 3)[RG.sample_index(W, H)][None]
    g.close()
    out = {"config": f"{name}.json {W}x{H} {spp} spp {b} bounces", "against": "unmodified reference, strict build (oracle/_ref/cray_ref_strict)",
           "sampled": f"{ref.shape[1]} fixed pixels (tests/reference_golden.py sample_index); x below is the sample's position"}
    out.update(compare_frames(gpu, ref))
    out["bound"] = rmse_bound(spp)
    out.update({"rays": int(st["rays"]), "gpu_seconds": round(time.time() - t0, 2)})
    record(out)
    assert out["nonfinite_gpu_only"] == [] and out["nonfinite_gpu"] <= out["nonfinite_reference"], out
    assert out["rmse"] <= out["bound"], out
