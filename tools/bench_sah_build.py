"""Device-built SAH trees (ptb_bvh_params.builder = PTB_BUILDER_SAH): build time against the host SAH build and the device LBVH,
and what the better tree buys the C5 path workload under the current kernels.

    python tools/bench_sah_build.py OUT_DIR [--reps 5] [--only c5,c8m] [--render-reps 5]

Scenes (records made once on the host, uploaded once into CUDA tensors before timing):
    c5   tessellate(cornell, 236): 2,005,056 triangles, the bench's C5 scene
    c8m  tessellate(cornell, 472): 8,020,224 triangles
Routes, each to a scene ready to render (every call ends in a synchronise, so a host clock around it measures the route):
    host_sah    ptb_scene_create on host records (the single-threaded host SAH build, then the upload)
    device_lbvh ptb_scene_create_from_device on the tensors, builder = PTB_BUILDER_LBVH
    device_sah  ptb_scene_create_from_device on the tensors, builder = PTB_BUILDER_SAH
One warm-up build per route, then --reps rounds that alternate the three routes; the reported time is the median.  Before
timing, the device SAH tree must equal the host tree byte for byte (ptb_scene_info, nodes, tri_order, quantised nodes and grid).
On c5, one PATH frame (3840x2160, depth 8, one sample) from each SAH scene must be identical bytes, and the LBVH and SAH
scenes are rendered alternately (--render-reps PATH frames each, same kernel and settings): Grays/s from the counters over a
host clock around the synchronised render, and node visits per ray from the counters of one more frame with statistics on.  Card name and power limit are read in
the same run.  Writes OUT_DIR/bench_sah_build.json.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_scene_build import card_info  # noqa: E402

SCENES = {"c5": 236, "c8m": 472}
W, H = 3840, 2160


def tree_bytes(sc):
    nodes, order = sc.bvh()
    q, lo, step = sc.bvh_quantized()
    return sc.info(), nodes.tobytes(), order.tobytes(), q.tobytes(), np.float32(lo + step).tobytes()


def run(out_dir, reps=5, only=("c5", "c8m"), render_reps=5):
    import torch

    import oclpathtracer_b200 as pt

    torch.cuda.init()
    dev = pt.Device(0, stream=torch.cuda.current_stream().cuda_stream)
    tris, mats = pt.load_model(os.path.join(ROOT, "data", "cornellbox.bin"))
    mats_t = torch.from_numpy(np.ascontiguousarray(mats).view(np.float32).reshape(-1, 16)).cuda()
    res = {"info": card_info(), "device": dev.name(), "reps": reps, "scenes": {}}
    sah = pt.bvh_params(builder=pt.BUILDER_SAH)

    for name in only:
        big = pt.tessellate(tris, SCENES[name])
        tris_t = torch.from_numpy(np.ascontiguousarray(big).view(np.float32).reshape(-1, 16)).cuda()
        torch.cuda.synchronize()

        def timed(fn):
            t0 = time.perf_counter()
            sc = fn()
            torch.cuda.synchronize()
            return sc, (time.perf_counter() - t0) * 1e3

        routes = {
            "host_sah": lambda: dev.scene(big, mats),
            "device_lbvh": lambda: dev.scene_from_device(tris_t, mats_t),
            "device_sah": lambda: dev.scene_from_device(tris_t, mats_t, sah),
        }
        # warm-up; the device SAH tree is the host tree
        scenes = {r: timed(fn)[0] for r, fn in routes.items()}
        host_tree = tree_bytes(scenes["host_sah"])
        assert tree_bytes(scenes["device_sah"]) == host_tree, name
        entry = {"triangles": len(big), "sah_tree_bytes_identical": True, "n_nodes_sah": host_tree[0]["n_nodes"],
                 "depth_sah": host_tree[0]["depth"], "n_nodes_lbvh": scenes["device_lbvh"].info()["n_nodes"],
                 "depth_lbvh": scenes["device_lbvh"].info()["depth"]}
        if name == "c5":
            frames = []
            prm = pt.default_params(width=W, height=H, n_frames=1, mode=pt.MODE_PATH, accum=pt.ACCUM_LINEAR, max_depth=8)
            for r in ("host_sah", "device_sah"):
                fb = dev.buffer(W * H * 16)
                dev.render(scenes[r], prm, fb)
                frames.append(fb.read(np.uint32).tobytes())
                fb.close()
            assert frames[0] == frames[1]
            entry["c5_frame_bytes_identical"] = True
            # the render gap: same kernel, same settings, LBVH against SAH, alternated
            fb = dev.buffer(W * H * 16)
            gap = {"device_lbvh": [], "device_sah": []}
            counters = {}
            for it in range(render_reps + 1):
                for r in gap:
                    prm = pt.default_params(width=W, height=H, first_frame=it, n_frames=1, mode=pt.MODE_PATH,
                                            accum=pt.ACCUM_LINEAR, max_depth=8)
                    dev.sync()
                    t0 = time.perf_counter()
                    ctr = dev.render(scenes[r], prm, fb, want_counters=True)
                    dev.sync()
                    secs = time.perf_counter() - t0
                    rays = ctr["rays_closest"] + ctr["rays_any"]
                    if it:  # the first round warms up
                        gap[r].append(rays / secs / 1e9)
            # node visits and triangle tests per ray: one more frame of each with statistics collected (not timed)
            sb = dev.buffer(W * H * 32)
            for r in gap:
                prm = pt.default_params(width=W, height=H, n_frames=1, mode=pt.MODE_PATH, accum=pt.ACCUM_LINEAR, max_depth=8,
                                        collect_stats=1)
                counters[r] = dev.render(scenes[r], prm, fb, sb, want_counters=True)
            sb.close()
            fb.close()
            entry["c5_path_4k_depth8"] = {
                r: {"grays_per_s": gap[r], "grays_per_s_median": float(np.median(gap[r])),
                    "nodes_per_ray": counters[r]["nodes"] / (counters[r]["rays_closest"] + counters[r]["rays_any"]),
                    "tri_tests_per_ray": counters[r]["tri_tests"] / (counters[r]["rays_closest"] + counters[r]["rays_any"]),
                    "counters": counters[r]} for r in gap}
            entry["c5_sah_over_lbvh_grays"] = (entry["c5_path_4k_depth8"]["device_sah"]["grays_per_s_median"]
                                               / entry["c5_path_4k_depth8"]["device_lbvh"]["grays_per_s_median"])
        for sc in scenes.values():
            sc.close()
        times = {r: [] for r in routes}
        for _ in range(reps):
            for r, fn in routes.items():
                sc, ms = timed(fn)
                sc.close()
                times[r].append(ms)
        entry["build_ms"] = times
        entry["build_median_ms"] = {r: float(np.median(v)) for r, v in times.items()}
        # where the device SAH build's time goes: device time of every kernel and copy of one build (a run of its own)
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CPU, torch.profiler.ProfilerActivity.CUDA]) as prof:
            routes["device_sah"]().close()
        rows = {}
        for ev in prof.key_averages():
            us = getattr(ev, "device_time_total", None)
            if us is None:
                us = ev.cuda_time_total
            if us > 0:
                rows[ev.key] = round(float(us) / 1e3, 4)
        entry["device_sah_device_time_ms"] = dict(sorted(rows.items(), key=lambda kv: -kv[1]))
        print(name, json.dumps({k: v for k, v in entry.items() if k not in ("build_ms", "device_sah_device_time_ms")}), flush=True)
        print(name, "device time of one device SAH build (ms):", json.dumps(entry["device_sah_device_time_ms"]), flush=True)
        res["scenes"][name] = entry
        del tris_t
        torch.cuda.empty_cache()
    dev.close()
    os.makedirs(out_dir, exist_ok=True)
    with open(os.path.join(out_dir, "bench_sah_build.json"), "w") as f:
        json.dump(res, f, indent=1)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--only", default="c5,c8m")
    ap.add_argument("--render-reps", type=int, default=5)
    a = ap.parse_args()
    res = run(a.out_dir, a.reps, tuple(a.only.split(",")), a.render_reps)
    print(json.dumps(res["info"]))


if __name__ == "__main__":
    main()
