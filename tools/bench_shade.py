"""Rates of ptb_scene_shade (Device.shade) against ptb_render on the same samples.

    python tools/bench_shade.py OUT_DIR [--reps 3] [--frames 16] [--only c5,c4,c2]

Workloads (the render's own camera rays and post-camera seeds of frames 0..frames-1, from ptb_test_camera, uploaded once):
    c5  tessellate(k=236) of the Cornell box (2,005,056 triangles, quantised binary nodes), PATH depth 8, 3840x2160
    c4  the Cornell box (FLAT form), PATH depth 8, 3840x2160
    c2  the Cornell box, AO with 16 rays, 1024x1024
The render runs all frames in one call (accum LINEAR), its time is the integrator time of ptb_device_profile (the resolve kernel
excluded); the shade call runs the same frames x pixels samples as one ray batch, timed with CUDA events.  Rounds alternate
render and shade, a 256 MiB buffer is overwritten before every timed call, and each rate is the median over --reps rounds.
Grays/s = (closest + any-hit queries from the counters) / time.  Before timing, the script asserts that the shade radiance
of every frame equals, bit for bit, the samples ptb_render writes for that frame alone (one frame, accum LINEAR).  Card name
and power limit are read in the same run.  Writes OUT_DIR/bench_shade.json.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "c5": dict(tess=236, mode=3, w=3840, h=2160, max_depth=8, ao_samples=16),
    "c4": dict(tess=0, mode=3, w=3840, h=2160, max_depth=8, ao_samples=16),
    "c2": dict(tess=0, mode=1, w=1024, h=1024, max_depth=16, ao_samples=16),
}


def card_info():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    if q.returncode != 0:
        return {"card": None, "note": "nvidia-smi unavailable"}
    name, power, clk = [x.strip() for x in q.stdout.strip().splitlines()[0].split(",")]
    return {"card": name, "power_limit": power, "sm_max_clock": clk}


def camera_samples(torch, dev, w, h, frames):
    """(frames * w * h, 8) int32 ptb_sample_ray records of the render's camera: frame-major, pixel order within a frame"""
    n = w * h
    rays = torch.zeros((frames * n, 8), dtype=torch.int32, device="cuda")
    gids = np.arange(n, dtype=np.int32)
    rec = np.zeros((n, 8), np.int32)
    for f in range(frames):
        o, d, s = dev.test_camera(w, h, f, gids)
        rec[:, 0:3] = o.view(np.int32)
        rec[:, 3] = s.view(np.int32)
        rec[:, 4:7] = d.view(np.int32)
        rays[f * n:(f + 1) * n].copy_(torch.from_numpy(rec))
    return rays


def run(out_dir, reps=3, frames=16, only=("c5", "c4", "c2")):
    import torch

    import oclpathtracer_b200 as pt

    torch.cuda.init()
    stream = torch.cuda.current_stream()
    dev = pt.Device(0, stream=stream.cuda_stream)
    tris, mats = pt.load_model(os.path.join(ROOT, "data", "cornellbox.bin"))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    res = {"info": card_info(), "frames": frames, "reps": reps, "workloads": {}}
    for name in only:
        wl = WORKLOADS[name]
        w, h = wl["w"], wl["h"]
        n = w * h * frames
        sc = dev.scene(pt.tessellate(tris, wl["tess"]) if wl["tess"] else tris, mats)
        prm = pt.default_params(width=w, height=h, first_frame=0, n_frames=frames, mode=wl["mode"], accum=pt.ACCUM_LINEAR,
                                max_depth=wl["max_depth"], ao_samples=wl["ao_samples"])
        rays = camera_samples(torch, dev, w, h, frames)
        rad = torch.empty((n, 4), dtype=torch.float32, device="cuda")
        frame = dev.buffer(w * h * 16)
        # the same samples: shade radiance of frame f == ptb_render of frame f alone
        _, ctr_s = dev.shade(sc, prm, rays, rad, want_counters=True)
        one = torch.empty((w * h, 4), dtype=torch.float32, device="cuda")
        fb1 = dev.wrap(one.data_ptr(), w * h * 16)
        for f in range(frames):
            p1 = pt.default_params(width=w, height=h, first_frame=f, n_frames=1, mode=wl["mode"], accum=pt.ACCUM_LINEAR,
                                   max_depth=wl["max_depth"], ao_samples=wl["ao_samples"])
            dev.render(sc, p1, fb1)
            dev.sync()
            assert torch.equal(one.view(torch.int32), rad[f * w * h:(f + 1) * w * h].view(torch.int32)), (name, f)
        fb1.close()
        ctr_r = dev.render(sc, prm, frame, want_counters=True)
        for k in ("rays_closest", "rays_any", "samples"):
            assert ctr_r[k] == ctr_s[k], (name, k, ctr_r[k], ctr_s[k])
        queries = ctr_r["rays_closest"] + ctr_r["rays_any"]
        dev.profile(True)
        dev.profile_read()
        r_ms, s_ms = [], []
        for rep in range(reps):
            flush.fill_(rep & 255)
            dev.render(sc, prm, frame)
            r_ms.append(dev.profile_read()["integrator_ms"])
            flush.fill_((rep + 1) & 255)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            dev.shade(sc, prm, rays, rad)
            b.record(stream)
            torch.cuda.synchronize()
            s_ms.append(a.elapsed_time(b))
        dev.profile(False)
        rr, sr = [queries / (ms * 1e-3) / 1e9 for ms in r_ms], [queries / (ms * 1e-3) / 1e9 for ms in s_ms]
        entry = {"scene_tris": int(sc.info()["n_tris"]), "mode": wl["mode"], "size": [w, h], "samples": n, "queries": queries,
                 "rays_bytes": n * 32, "bit_identical_to_render": True,
                 "render_integrator_ms": r_ms, "shade_ms": s_ms,
                 "render_grays_s": float(np.median(rr)), "shade_grays_s": float(np.median(sr)),
                 "shade_over_render": float(np.median(sr) / np.median(rr))}
        print(name, json.dumps(entry), flush=True)
        res["workloads"][name] = entry
        frame.close()
        del rays, rad, one
        torch.cuda.empty_cache()
        sc.close()
    dev.close()
    os.makedirs(out_dir, exist_ok=True)
    with open(os.path.join(out_dir, "bench_shade.json"), "w") as f:
        json.dump(res, f, indent=1)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--frames", type=int, default=16)
    ap.add_argument("--only", default="c5,c4,c2")
    a = ap.parse_args()
    res = run(a.out_dir, a.reps, a.frames, tuple(a.only.split(",")))
    print(json.dumps(res["info"]))


if __name__ == "__main__":
    main()
