"""Rates of ptb_scene_intersect (Device.intersect) on caller-owned device ray buffers.

    python tools/bench_intersect.py OUT_DIR [--reps 5] [--window 0.25] [--log2n 24]

Scenes: C5 (tessellate(k=236) of the Cornell box: 2,005,056 triangles, host SAH build, quantised binary nodes) and the Cornell
box itself (FLAT form).  Ray sets, all generated from fixed seeds:
    incoherent  2^24 rays, origins uniform in the scene's box, directions uniform on the sphere   (closest hit)
    coherent    the camera rays of frame 0 of a 3840x2160 image (ptb_test_camera), uploaded      (closest hit)
    shadow      the incoherent set with tmax uniform in (0, 3]                                    (any hit)
Each rate is the median over --reps repetitions of CUDA-event time over a window of >= --window seconds of back-to-back calls;
a 256 MiB buffer is overwritten before every repetition so that no ray, node or triangle starts in L2.  As an A/B on the same
rays, the k_trace kernel time of one ptb_trace call (the parity-test hook: one thread per ray, no dynamic fetch) is taken from a
separate torch.profiler run (kernel time only, its host copies excluded).  Card name and power limit are read in the same run.
Writes OUT_DIR/bench_intersect.json.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card_info():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    if q.returncode != 0:
        return {"card": None, "note": "nvidia-smi unavailable"}
    name, power, clk = [x.strip() for x in q.stdout.strip().splitlines()[0].split(",")]
    return {"card": name, "power_limit": power, "sm_max_clock": clk}


def incoherent_rays(torch, lo, hi, n, seed, shadow=False):
    """(n, 8) float32: origins uniform in [lo, hi], directions uniform on the sphere; tmax 1e20, or uniform in (0, 3]"""
    g = torch.Generator(device="cuda").manual_seed(seed)
    r = torch.zeros((n, 8), dtype=torch.float32, device="cuda")
    lo_t = torch.tensor(lo, dtype=torch.float32, device="cuda")
    hi_t = torch.tensor(hi, dtype=torch.float32, device="cuda")
    r[:, 0:3] = lo_t + (hi_t - lo_t) * torch.rand((n, 3), generator=g, device="cuda")
    d = torch.randn((n, 3), generator=g, device="cuda")
    r[:, 4:7] = d / d.norm(dim=1, keepdim=True)
    if shadow:
        r[:, 3] = 3.0 * (1.0 - torch.rand(n, generator=g, device="cuda"))  # (0, 3]
    else:
        r[:, 3] = 1e20
    return r


def camera_rays(torch, dev, w, h, frame=0):
    gids = np.arange(w * h, dtype=np.int32)
    o, d, _ = dev.test_camera(w, h, frame, gids)
    r = np.zeros((w * h, 8), np.float32)
    r[:, 0:3], r[:, 3], r[:, 4:7] = o, np.float32(1e20), d
    return torch.from_numpy(r).cuda()


def time_query(torch, dev, scene, rays, hits, any_hit, flush, reps, window):
    """median Grays/s over reps windows of >= `window` seconds of back-to-back calls"""
    stream = torch.cuda.current_stream()
    for _ in range(2):
        dev.intersect(scene, rays, hits, any_hit=any_hit)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    dev.intersect(scene, rays, hits, any_hit=any_hit)
    torch.cuda.synchronize()
    calls = max(1, int(np.ceil(window / max(time.perf_counter() - t0, 1e-6))))
    rates = []
    for rep in range(reps):
        flush.fill_(rep & 255)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for _ in range(calls):
            dev.intersect(scene, rays, hits, any_hit=any_hit)
        b.record(stream)
        torch.cuda.synchronize()
        ms = a.elapsed_time(b)
        rates.append(calls * rays.shape[0] / (ms * 1e-3) / 1e9)
    return {"grays_s": float(np.median(rates)), "min": float(min(rates)), "max": float(max(rates)), "calls_per_window": calls,
            "window_s": calls * rays.shape[0] / (float(np.median(rates)) * 1e9)}


def trace_kernel_rate(torch, dev, scene, rays, any_hit):
    """Grays/s of the k_trace kernel of one ptb_trace call on the same rays (kernel time from torch.profiler)"""
    from torch.profiler import ProfilerActivity, profile

    h = rays.cpu().numpy()
    o, tmax, d = h[:, 0:3].copy(), h[:, 3].copy(), h[:, 4:7].copy()
    dev.trace(scene, o, d, tmax, any_hit=any_hit)  # warm-up (module load, allocations)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        dev.trace(scene, o, d, tmax, any_hit=any_hit)
    us = sum(e.device_time_total for e in prof.key_averages() if "k_trace" in e.key)
    return {"grays_s": len(h) / (us * 1e-6) / 1e9 if us else None, "kernel_ms": us / 1e3}


def run(out_dir, reps=5, window=0.25, log2n=24, with_trace=True, scenes=("c5", "cornell")):
    import torch

    import oclpathtracer_b200 as pt

    torch.cuda.init()
    dev = pt.Device(0, stream=torch.cuda.current_stream().cuda_stream)
    tris, mats = pt.load_model(os.path.join(ROOT, "data", "cornellbox.bin"))
    pts = np.concatenate([tris["p1"][:, :3], tris["p2"][:, :3], tris["p3"][:, :3]])
    lo, hi = pts.min(0).tolist(), pts.max(0).tolist()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    n = 1 << log2n
    sets = {
        "incoherent": (incoherent_rays(torch, lo, hi, n, 1), False),
        "coherent": (camera_rays(torch, dev, 3840, 2160), False),
        "shadow": (incoherent_rays(torch, lo, hi, n, 1, shadow=True), True),
    }
    res = {"info": card_info(), "rays": {k: int(v[0].shape[0]) for k, v in sets.items()}, "scenes": {}}
    for name in scenes:
        t0 = time.perf_counter()
        sc = dev.scene(pt.tessellate(tris, 236) if name == "c5" else tris, mats)
        info = sc.info()
        entry = {"n_tris": info["n_tris"], "form": {1: "FLAT", 4: "4-wide", 2: "quantised binary"}[info["width"]],
                 "build_s": time.perf_counter() - t0, "sets": {}}
        for sname, (rays, any_hit) in sets.items():
            hits = torch.empty((rays.shape[0], 4), dtype=torch.float32, device="cuda")
            r = time_query(torch, dev, sc, rays, hits, any_hit, flush, reps, window)
            r["query"] = "any" if any_hit else "closest"
            hv = hits.view(torch.int32)[:, 3]
            r["hit_fraction"] = float((hv >= 0).float().mean())
            if with_trace:
                r["k_trace"] = trace_kernel_rate(torch, dev, sc, rays, any_hit)
            entry["sets"][sname] = r
            print(name, sname, json.dumps(r), flush=True)
        res["scenes"][name] = entry
        sc.close()
    dev.close()
    os.makedirs(out_dir, exist_ok=True)
    with open(os.path.join(out_dir, "bench_intersect.json"), "w") as f:
        json.dump(res, f, indent=1)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--window", type=float, default=0.25)
    ap.add_argument("--log2n", type=int, default=24)
    a = ap.parse_args()
    res = run(a.out_dir, a.reps, a.window, a.log2n)
    print(json.dumps(res["info"]))


if __name__ == "__main__":
    main()
