#!/usr/bin/env python3
"""bench.py — Mray/s (and Msample/s) of the B200 path-trace hot loop on BASELINE.json's headline config.

A "step" is one complete render of the workload frame: default = configs[1] of BASELINE.json,
input/hdr.json at 1920x1080, 1000 spp, 32 bounces; --workload refraction | venus | hdr8k are configs[2..4].
The tile grid of the host C dispatcher (quantizeImage) is dealt out to the ranks by a spatial interleave
((tx + 5 ty) % world, cr_renderer.c takeRankTiles); the frame is fixed, so this is STRONG scaling.  With N>1 the fp32
framebuffer tiles are gathered on rank 0 over NCCL (libcrgpu_nccl.so) inside the timed region.

  value      Mray/s, whole job, scene + framebuffer resident in HBM, device-timed (CUDA events), max over ranks;
             the tile gather of N>1 is the product's (libcrgpu_nccl.so, grouped ncclSend/ncclRecv) on the same stream
  e2e        same metric through the reference-facing C API with HOST buffers: libcrhost.so `renderFrame` (the host C
             mirror of c-ray's tile dispatcher) — H2D of the prepared scene from pinned host memory, tiles, NCCL gather
             in C, D2H of the fp32 renderBuffer + the 8-bit image — wall clock around the call, max over ranks.
             The scene is loaded from input/*.json by THIS repository's loader (libcrloader.so), once, like loadScene.
  roofline   K2 (k_trace) algorithmic bytes / its CUDA-event time, vs the measured HBM copy peak
  cpu_baseline  the UNMODIFIED reference (oracle/_ref/cray_ref_stock, pthreads, all host cores) on a bounded
             sample (same frame, fewer spp) — a reported baseline, not the optimisation target

`--impl reference` times that same reference binary as its own arm.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "c-ray_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

WORKLOADS = {   # BASELINE.json configs[0..4]
    "hdr": dict(scene="hdr", width=1920, height=1080, spp=1000, bounces=32),             # C2: the configuration the metric is quoted on (default)
    "refraction": dict(scene="refraction", width=1920, height=1080, spp=2500, bounces=512),   # C3
    "venus": dict(scene="venus", width=2560, height=1600, spp=1000, bounces=25),         # C4
    "hdr8k": dict(scene="hdr", width=7680, height=4320, spp=4000, bounces=32),           # C5: the 8-GPU frame (fits one GPU too; --spp reduces it)
    "scene": dict(scene="scene", width=320, height=200, spp=16, bounces=4),              # C1 geometry
}
PEAK_FALLBACK_GBS = 6650.0   # HBM copy bandwidth assumed when MEASURED_PEAKS.json is absent
DUMP_LIMIT_BYTES = 64 << 20   # --dump-outputs writes at most this much; a larger framebuffer is written as a fixed pixel sample


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="hdr", choices=sorted(WORKLOADS))
    ap.add_argument("--width", type=int, default=0)
    ap.add_argument("--height", type=int, default=0)
    ap.add_argument("--spp", type=int, default=0)
    ap.add_argument("--bounces", type=int, default=0)
    ap.add_argument("--tile", type=int, default=0, help="tile edge of the dispatcher's tile grid (default 64)")
    ap.add_argument("--max-paths", type=int, default=0, help="paths in flight per wavefront batch (0 = library default)")
    ap.add_argument("--cpu-spp", type=int, default=0, help="spp of the bounded CPU-baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ingest", action="store_true", help="skip the informational loader-vs-reference-loader timing")
    ap.add_argument("--crscene", action="store_true", help="take the scene from scenes/_built/*.crscene (reference loader's export) instead of parsing the JSON")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the fp32 framebuffer of the last timed step to DIR/framebuffer.npy, so that two builds can be compared")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    return args


def dump_outputs(directory, fb):
    """The framebuffer the timed path returned ((H, W, 3) float32).  Above DUMP_LIMIT_BYTES a fixed, seeded sample of pixels is
    written instead: framebuffer_sample.npy (n, 3) float32 and framebuffer_sample_pixels.npy (n,) float64 row-major pixel indices."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    if fb.nbytes <= DUMP_LIMIT_BYTES:
        np.save(os.path.join(directory, "framebuffer.npy"), fb)
        return
    pixels = fb.shape[0] * fb.shape[1]
    n = (DUMP_LIMIT_BYTES - 4096) // (3 * 4 + 8)     # (npy headers take the 4096)
    idx = np.sort(np.random.default_rng(0).choice(pixels, size=n, replace=False))
    np.save(os.path.join(directory, "framebuffer_sample.npy"), fb.reshape(pixels, 3)[idx])
    np.save(os.path.join(directory, "framebuffer_sample_pixels.npy"), idx.astype(np.float64))


def workload(args):
    w = dict(WORKLOADS[args.workload])
    for k, a in (("width", args.width), ("height", args.height), ("spp", args.spp), ("bounces", args.bounces)):
        if a > 0:
            w[k] = a
    return w


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"], "measured"
    except Exception:
        return PEAK_FALLBACK_GBS, "fallback"


class ClockSampler(threading.Thread):
    """SM clock + throttle reasons DURING the timed region, read through NVML in-process (spawning nvidia-smi
    every 200 ms measurably stalls kernel submission: it takes the driver lock for ~0.5 s per call)."""
    REASONS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.sm, self.mask, self.stop_flag, self.max_mhz, self.err = index, [], 0, False, None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and all(v.strip().isdigit() for v in vis.split(",")) else index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as e:   # noqa: BLE001
            self.nv, self.err = None, str(e)

    def run(self):
        if not self.nv:
            return
        while not self.stop_flag:
            try:
                self.sm.append(float(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)))
                self.mask |= int(self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
            except Exception as e:   # noqa: BLE001
                self.err = str(e)
            time.sleep(0.05)

    def summary(self):
        self.stop_flag = True
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml unavailable: %s" % self.err]}
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2], "sm_mhz_min": sm[0], "sm_max_mhz": self.max_mhz,
                "reasons": [n for n, bit in self.REASONS.items() if self.mask & bit], "samples": len(sm)}


def run_reference(scene, W, H, spp, bounces, threads):
    """The unmodified reference (stock flags, pthreads) on the host cores; returns (seconds of renderFrame, samples)."""
    exe = os.path.join(ROOT, "oracle", "_ref", "cray_ref_stock")
    js = os.path.join(ROOT, "oracle", "_ref", "input", scene + ".json")
    if not (os.path.exists(exe) and os.path.exists(js)):
        return None
    out = f"/tmp/cray_ref_bench_{os.getpid()}.f32"
    r = subprocess.run([exe, "render", js, str(W), str(H), str(spp), str(bounces), str(threads), "0", "0", out],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    try:
        os.remove(out)
    except OSError:
        pass
    m = re.search(r"REF_RENDER .*threads=(\d+) seconds=([0-9.]+)", r.stdout)
    if r.returncode != 0 or not m:
        return None
    return float(m.group(2)), W * H * spp, int(m.group(1))


def scene_ingest(scene):
    """SURVEY 8(f2), informational: JSON + OBJ/MTL + PNG/HDR + both BVH levels -> flat scene on the host cores,
    this repository's loader (libcrloader.so) next to the reference's own loader (oracle/_ref harness `export`)."""
    try:
        import crscene
        js = os.path.join(ROOT, "oracle", "_ref", "input", scene + ".json")
        if not os.path.exists(js):
            return None
        best = None
        for _ in range(3):
            t0 = time.perf_counter()
            flat = crscene.load_json(js)
            dt = time.perf_counter() - t0
            polys, nodes = int(flat.poly_count), int(flat.bvh_node_count)
            crscene.free(flat)
            best = dt if best is None else min(best, dt)
        out = {"loader_s": round(best, 3), "threads": os.cpu_count() or 1, "triangles": polys, "bvh_nodes": nodes,
               "what": f"crloader_load_json(input/{scene}.json): parse + decode + SAH BVH build, best of 3"}
        exe = os.path.join(ROOT, "oracle", "_ref", "cray_ref_stock")
        if os.path.exists(exe):
            tmp = f"/tmp/cray_ref_ingest_{os.getpid()}.crscene"
            t0 = time.perf_counter()
            r = subprocess.run([exe, "export", js, "0", "0", "0", "0", tmp], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            dt = time.perf_counter() - t0
            if r.returncode == 0:
                out["reference_s"] = round(dt, 3)
                out["reference_what"] = "unmodified reference loader (process start + loadScene + flatten + write), one run"
            try:
                os.remove(tmp)
            except OSError:
                pass
        return out
    except Exception as e:      # informational only: never fail the bench line
        return {"error": str(e)[:200]}


def reference_arm(args, w, rank):
    """bench.py --impl reference: the reference's own CPU implementation of the path, rank 0 only."""
    if rank != 0:
        return
    cores = usable_threads()
    spp = args.cpu_spp or max(1, min(w["spp"], int(5.0e7 / (w["width"] * w["height"])) or 1))   # a few seconds of CPU rendering per step
    rays_per_sample = float(os.environ.get("CRAY_RAYS_PER_SAMPLE", "0")) or None
    times = []
    for i in range(args.warmup + args.steps):
        r = run_reference(w["scene"], w["width"], w["height"], spp, w["bounces"], cores)
        if r is None:
            print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/cray_ref_stock or its input assets are missing (run build() in the build container)"}))
            return
        if i >= args.warmup:
            times.append(r[0])
        threads = r[2]
    total_s = sum(times)
    samples = w["width"] * w["height"] * spp * args.steps
    msample = samples / total_s / 1e6
    # the reference never counts rays (SURVEY §6); rays/sample of the same scene+bounces is measured by the oracle port
    rps = rays_per_sample or oracle_rays_per_sample(w, spp)
    value = msample * rps
    line = {"metric": "Mray/s", "value": round(value, 3), "unit": "Mray/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(1e3 * total_s / args.steps, 3), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "bundled scene input/%s.json (reference assets copied at build time)" % w["scene"], "impl": "reference",
            "config": {"workload": f"input/{w['scene']}.json {w['width']}x{w['height']} {w['spp']} spp {w['bounces']} bounces", "name": args.workload, "spp_per_step": spp,
                       "note": "bounded sample: same frame, fewer spp (CPU cost is linear in spp, renderer.c:275)"},
            "msample_per_s": round(msample, 3), "rays_per_sample": round(rps, 4),
            "cpu_baseline": {"value": round(value, 3), "unit": "Mray/s", "cores": threads, "kind": "reference", "host": host_cpus(),
                             "sample": f"{w['width']}x{w['height']} x {spp} spp per step, pthreads -j {threads}, stock flags (-O2 -ftree-vectorize -march=x86-64-v3)"},
            "e2e": {"value": round(value, 3), "unit": "Mray/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def oracle_rays_per_sample(w, spp):
    """rays per pathTrace call for this scene/bounce limit, counted by the CPU oracle on a small frame."""
    import oracle_lib as O
    sw, sh = max(16, w["width"] // 8), max(16, w["height"] // 8)
    o = O.OracleScene(os.path.join(ROOT, "scenes", "_built", w["scene"] + ".crscene"), sw, sh, max(1, min(spp, 4)), w["bounces"])
    _, c = o.render(threads=os.cpu_count() or 1, count=True)
    o.close()
    return c["rays"] / c["paths"]


def host_cpus():
    """What this process may actually use: os.cpu_count() is the machine, not the cgroup/affinity share (a 5x swing of the CPU
    arm between two boxes that both 'have 128 cores' was exactly that)."""
    out = {"cpu_count": os.cpu_count() or 1}
    try:
        out["affinity"] = len(os.sched_getaffinity(0))
    except Exception:   # noqa: BLE001
        pass
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            out["cgroup_" + os.path.basename(path)] = open(path).read().strip()
            break
        except OSError:
            continue
    try:
        out["loadavg_1m"] = round(os.getloadavg()[0], 1)
    except OSError:
        pass
    return out


def usable_threads():
    h = host_cpus()
    n = h.get("affinity", h["cpu_count"])
    q = h.get("cgroup_cpu.max", "")
    m = re.match(r"(\d+)\s+(\d+)", q)
    if m and int(m.group(2)) > 0:
        n = max(1, min(n, int(int(m.group(1)) / int(m.group(2)) + 0.5)))
    return n


def main():
    args = parse_args()
    w = workload(args)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        reference_arm(args, w, rank)
        return

    # rank 0 prints ONE JSON line on stdout and nothing else: NCCL announces "NCCL version ..." on fd 1 when the first communicator is
    # created (torch's and libcrgpu_nccl's), so fd 1 points at stderr for the whole run and the line goes to the saved descriptor
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    import zlib
    import numpy as np
    import torch
    import crgpu
    import crhost

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the hot path has no CPU fallback")
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    work_stream = torch.cuda.Stream(device=dev)      # library kernels, the C NCCL gather and the timing events all live on this stream
    torch.cuda.set_stream(work_stream)

    W, H, spp, bounces = w["width"], w["height"], w["spp"], w["bounces"]
    tile = args.tile if args.tile > 0 else 64       # the tile dispatcher's grid (tile-ordered pixel lists keep warps on compact 2D footprints)

    # ---- the scene: input/<scene>.json through THIS repository's loader (SURVEY 8 f2), like loadScene: once, outside the frames
    refdir = os.path.join(ROOT, "oracle", "_ref")
    js = os.path.join("input", w["scene"] + ".json")
    flat_fallback = os.path.join(ROOT, "scenes", "_built", w["scene"] + ".crscene")
    t_in = time.perf_counter()
    if os.path.exists(os.path.join(refdir, js)) and not args.crscene:
        cwd = os.getcwd()
        os.chdir(refdir)                   # node-graph texture paths are relative to the reference's working directory (sceneloader.c:783)
        try:
            R = crhost.Renderer(js, W, H, spp, bounces, gpus=1, tile=tile, quiet=True)
        finally:
            os.chdir(cwd)
        scene_src = f"input/{w['scene']}.json parsed + BVH-built by libcrloader.so (this repository's loader)"
    elif os.path.exists(flat_fallback):
        R = crhost.Renderer(flat_fallback, W, H, spp, bounces, gpus=1, tile=tile, quiet=True)
        scene_src = f"scenes/_built/{w['scene']}.crscene (flattened by the reference loader at build time)"
    else:
        raise SystemExit("no scene: neither oracle/_ref/input nor scenes/_built present — run __graft_entry__.build() in the build container")
    ingest_s = time.perf_counter() - t_in

    # ---- the GPU group: rank 0 makes the NCCL id, torch.distributed (the launcher's plumbing) hands it out, the C host joins
    if world > 1:
        box = [crhost.unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        R.join(box[0], rank, world, local)
    else:
        R.join(None, 0, 1, local)
    t_p = time.perf_counter()
    R.prepare()                                   # re-layout for the kernels into pinned host memory (part of scene loading)
    prepare_s = time.perf_counter() - t_p
    my_rects, owner, all_rects = R.rank_tiles(rank, world)

    # ---- value: scene + framebuffer resident, device-timed ------------------------------------------------------------------
    g = crgpu.GpuScene(None, samples=spp, bounces=bounces, device=local, max_paths=args.max_paths or None, prepared=R.prepared())
    gather = None
    if world > 1:
        gather = crgpu.RankGather(R.comm())
        gather.set_stream(torch.cuda.current_stream(dev).cuda_stream)

    def step(flags=0):
        """one complete frame: everything enqueued on torch's current stream"""
        g.clear()
        g.render_tiles(my_rects, flags=flags | crgpu.FLAG_ASYNC)       # the rank's whole share of the tile grid as one wavefront
        if gather:
            gather.gather(g, all_rects, owner, 0)

    def barrier():
        torch.cuda.synchronize(dev)
        if dist:
            dist.barrier()
        torch.cuda.synchronize(dev)

    g.set_stream(torch.cuda.current_stream(dev).cuda_stream)
    for _ in range(args.warmup):
        step()
    g.get_stats()
    sampler = ClockSampler(local)
    sampler.start()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    wall0 = time.perf_counter()
    ev0.record()
    for i in range(args.steps):
        step()
    ev1.record()
    barrier()
    wall_ms = 1e3 * (time.perf_counter() - wall0)
    ms = ev0.elapsed_time(ev1)
    if ms < 0.9 * wall_ms:      # events that do not bracket the kernels (wrong stream) must never flatter the number
        sys.stderr.write(f"bench.py: CUDA-event time {ms:.1f} ms << wall {wall_ms:.1f} ms; reporting wall clock\n")
        ms = wall_ms
    stats = g.get_stats()
    clocks = sampler.summary()
    last_fb = g.read() if rank == 0 else None     # rank 0 holds the gathered frame of the last timed step
    value_crc = zlib.crc32(last_fb.tobytes()) if rank == 0 else 0
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, last_fb)
    tms = torch.tensor([ms, float(stats["rays"]), float(stats["paths"]), float(stats["kernel_launches"])], device=dev, dtype=torch.float64)
    rank_ms = [float(tms[0])]
    if dist:
        allms = [torch.zeros(1, device=dev, dtype=torch.float64) for _ in range(world)]
        dist.all_gather(allms, tms[:1].clone())
        rank_ms = [round(float(x[0]) / args.steps, 3) for x in allms]     # per-rank device time per step: tile imbalance shows here
        mx = tms.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = tms.clone()
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        ms, rays, paths, launches = float(mx[0]), float(sm[1]), float(sm[2]), float(sm[3])
    else:
        ms, rays, paths, launches = float(tms[0]), float(tms[1]), float(tms[2]), float(tms[3])
    value = rays / ms / 1e3                      # Mray/s, whole job
    msample = paths / ms / 1e3

    # ---- roofline of K2 / K3: one profiled step (per-kernel CUDA events) + one counted step (P/T/S/I) ---------------
    if gather:
        gather.use_own_stream()
    g.use_own_stream()
    g.clear()
    prof = g.render_tiles(my_rects, flags=crgpu.FLAG_TIME_KERNELS)
    cspp = min(spp, 8)
    g.clear()
    cnt = g.render_tiles(my_rects, pass_begin=0, pass_count=cspp, flags=crgpu.FLAG_COUNT)
    g.close()
    P, T, S, I = (cnt[k] / cnt["rays"] for k in ("node_pairs", "tri_tests", "sphere_tests", "inst_visits"))
    b_ray = 64 * P + 80 * T + 128 * I + 16 * S + 72          # SURVEY.md §8(d)
    peak, peak_kind = peaks()
    trace_s = prof["trace_ms"] / 1e3
    shade_s = prof["shade_ms"] / 1e3
    achieved = (prof["rays"] * b_ray / trace_s / 1e9) if trace_s > 0 else None
    traffic, traffic_note, issue = None, None, None
    try:   # DRAM bytes of one K2 launch from the committed ncu --set full capture (not live: ncu replays kernels ~40x)
        import glob
        mfile = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_metrics.json")))[-1]
        m = json.load(open(mfile))["kernels"]["k_trace"][0]
        traffic = int((m["dram_read"] + m["dram_write"]) * 1e9)
        issue = {"active_threads_per_warp_inst": round(m["active_threads_per_warp_inst"], 2), "issue_active_pct": round(m["issue_active_pct"], 1),
                 "warps_active_pct": round(m["warps_active_pct"], 1),
                 "dram_gbs": round((m["dram_read"] + m["dram_write"]) / (m["duration"] / 1e3), 1),
                 "note": "what actually limits k_trace (same ncu capture): instruction issue at ~half the SIMT lanes, not DRAM"}
        traffic_note = (f"{os.path.basename(mfile)}: k_trace bounce-1 launch of a 66M-path batch on input/hdr.json ({m['duration']:.2f} ms): "
                        f"{traffic / 1e9:.2f} GB of DRAM traffic, far BELOW the algorithmic figure because nodes and triangles are served by L1/L2")
    except Exception:   # noqa: BLE001
        pass
    shade_bytes = 116.0    # K3 per ray: 68 B in (ray 48 + hit 20) + 48 B out when the path survives (DESIGN.md §4)
    roofline = {"bound": "hbm", "kernel": "k_trace", "achieved": round(achieved, 2) if achieved else None, "peak": peak,
                "peak_kind": peak_kind + " HBM copy bandwidth (MEASURED_PEAKS.json)" if peak_kind == "measured" else "fallback 6.65 TB/s",
                "unit": "GB/s", "frac": round(achieved / peak, 4) if achieved else None, "traffic": traffic, "traffic_note": traffic_note, "sm_issue": issue,
                "bytes_per_ray": round(b_ray, 1), "per_ray": {"P": round(P, 3), "T": round(T, 3), "I": round(I, 3), "S": round(S, 3)},
                "trace_share_of_step": round(prof["trace_ms"] / prof["total_ms"], 4) if prof["total_ms"] else None,
                "shade_share_of_step": round(prof["shade_ms"] / prof["total_ms"], 4) if prof["total_ms"] else None,
                "trace_gray_per_s": round(prof["rays"] / trace_s / 1e9, 3) if trace_s > 0 else None,
                "shade": {"kernel": "k_shade (+k_bucket)", "bytes_per_ray": shade_bytes, "gray_per_s": round(prof["rays"] / shade_s / 1e9, 3) if shade_s > 0 else None,
                          "achieved": round(prof["rays"] * shade_bytes / shade_s / 1e9, 2) if shade_s > 0 else None,
                          "frac": round(prof["rays"] * shade_bytes / shade_s / 1e9 / peak, 4) if shade_s > 0 else None},
                "note": "achieved = rays * B_ray / sum of k_trace launch durations (CUDA events, rank-local profiled step); "
                        "the scene (~50 MB) is L2-resident, so DRAM traffic is mostly the wavefront state"}

    # ---- e2e: libcrhost.so renderFrame, host scene -> host frame, wall clock --------------------------------------------------
    e_steps = args.steps
    R.render()                                   # one untimed frame: first-touch of this process' renderFrame path (threads, caches)
    barrier()
    t0 = time.perf_counter()
    e_rays = 0
    for _ in range(e_steps):
        _, r_ = R.render()
        e_rays += r_
    barrier()
    e_ms = 1e3 * (time.perf_counter() - t0)
    fb = R.framebuffer()
    frame_crc = zlib.crc32(fb.tobytes()) if rank == 0 else 0
    finite = bool(np.isfinite(fb).all()) if rank == 0 else True
    et = torch.tensor([e_ms, float(e_rays)], device=dev, dtype=torch.float64)
    if dist:
        a = et.clone(); dist.all_reduce(a, op=dist.ReduceOp.MAX)
        b = et.clone(); dist.all_reduce(b, op=dist.ReduceOp.SUM)
        e_ms, e_rays = float(a[0]), float(b[1])
    e2e_value = e_rays / e_ms / 1e3
    h2d = 0
    try:
        import ctypes as C
        n = C.c_size_t()
        crgpu.lib().crgpu_prepared_slab.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_size_t)]
        crgpu.lib().crgpu_prepared_slab(C.c_void_p(R.prepared()), None, C.byref(n))
        h2d = int(n.value)
    except Exception:   # noqa: BLE001
        pass
    R.close()

    # ---- CPU baseline: the unmodified reference on the host cores, bounded sample, rank 0 at N=1 ------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = usable_threads()
        cspp = args.cpu_spp or max(1, min(spp, int(2.5e8 / (W * H)) or 1))   # ~10-30 s of CPU rendering (5-15 Msample/s on the host)
        r = run_reference(w["scene"], W, H, cspp, bounces, cores)
        if r:
            secs, samples, threads = r
            cpu = {"value": round(samples / secs / 1e6 * (rays / paths), 3), "unit": "Mray/s", "cores": threads, "kind": "reference",
                   "msample_per_s": round(samples / secs / 1e6, 3), "seconds": round(secs, 2), "host": host_cpus(),
                   "sample": f"unmodified reference (oracle/_ref/cray_ref_stock, pthreads -j {threads}) on input/{w['scene']}.json {W}x{H}, "
                             f"{cspp} spp of {spp}, {bounces} bounces; Mray/s = its Msample/s x {rays / paths:.3f} rays/sample counted on the GPU run"}
        else:
            cpu = {"value": None, "unit": "Mray/s", "cores": cores, "kind": "reference", "sample": "oracle/_ref missing", "host": host_cpus()}

    if rank == 0:
        line = {"metric": "Mray/s", "value": round(value, 2), "unit": "Mray/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": round(ms / args.steps, 3), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f32", "data": "bundled scene " + scene_src + " (no synthetic tensors on this path)",
                "config": {"workload": f"input/{w['scene']}.json {W}x{H} {spp} spp {bounces} bounces", "name": args.workload, "tile": tile,
                           "parallelism": f"tile-sharded x{world} (tile (tx + 5 ty) % world), one NCCL gather per frame" if world > 1 else "1 GPU",
                           "l2": "wavefront state (GBs per step) streams through the 126 MB L2: inputs larger than L2, no explicit flush"},
                "msample_per_s": round(msample, 2), "rays_per_sample": round(rays / paths, 4), "rank_ms_per_step": rank_ms if world > 1 else None,
                "e2e": {"value": round(e2e_value, 2), "unit": "Mray/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": H * W * 3 * 4 + H * W * 3,
                        "ms_per_step": round(e_ms / e_steps, 3), "steps": e_steps,
                        "what": "libcrhost.so renderFrame: prepared scene (pinned host) -> H2D -> tiles through the C dispatcher -> NCCL gather (C) -> "
                                "D2H fp32 renderBuffer + 8-bit sRGB image (host)"},
                "frame_crc32": f"{frame_crc:08x}", "value_path_crc32": f"{value_crc:08x}", "frame_finite": finite,
                "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline,
                "scene_load": {"loader_s": round(ingest_s, 3), "prepare_s": round(prepare_s, 3),
                               "what": "crloader_load_json (parse + decode + both BVH levels) and crgpu_prepare (re-layout into pinned memory); once per scene, outside the frames"}}
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if world == 1 and not args.no_cpu_baseline and not args.no_ingest:
            ingest = scene_ingest(w["scene"])
            if ingest:
                line["scene_ingest"] = ingest
        sys.stdout.flush()
        os.write(real_stdout, (json.dumps(line) + "\n").encode())
    if dist:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
