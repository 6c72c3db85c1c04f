"""Time to a ready LBVH scene from triangle records that live in a CUDA tensor: the host route against the device route.

    python tools/bench_scene_build.py OUT_DIR [--reps 7] [--only c5,c8m]

Scenes (records made once on the host, uploaded once into CUDA tensors before timing):
    c5   tessellate(cornell, 236): 2,005,056 triangles, the bench's C5 scene
    c8m  tessellate(cornell, 472): 8,020,224 triangles
Routes, each from the tensors to a scene ready to render:
    host    tensor.cpu() of the triangle and material records, then ptb_scene_create_gpu (host checks, upload, device build)
    device  ptb_scene_create_from_device on the tensors (Device.scene_from_device)
Both calls end in a synchronise (ptb_scene_create_gpu and ptb_scene_create_from_device return when the scene is ready; the
script also synchronises torch's stream), so a host clock around them measures the whole route.  One warm-up build per route,
then --reps rounds that alternate the two routes in this process; the reported time is the median.  The host route is also
split into its download (tensor.cpu()) and its ptb_scene_create_gpu call.  Before timing, the two scenes' trees are compared
(info, live nodes, tri_order) and one PATH frame of the C5 workload (3840x2160, depth 8, one sample) rendered from each must be
identical bytes.  A separate torch.profiler pass (CUDA activities) over one build of each route lists the device time of
every kernel and copy, so the difference between the routes can be attributed.  Card name and power limit are read in the
same run.  Writes OUT_DIR/bench_scene_build.json.
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

SCENES = {"c5": 236, "c8m": 472}


def card_info():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    if q.returncode != 0:
        return {"card": None, "note": "nvidia-smi unavailable"}
    name, power, clk = [x.strip() for x in q.stdout.strip().splitlines()[0].split(",")]
    return {"card": name, "power_limit": power, "sm_max_clock": clk}


def live_nodes(nodes):
    live = np.zeros(len(nodes), bool)
    front = np.array([0])
    while front.size:
        live[front] = True
        ch = np.concatenate([nodes["child0"][front], nodes["child1"][front]])
        front = ch[(ch >= 0) & (ch != 0x7FFFFFFF)]
    return live


def run(out_dir, reps=7, only=("c5", "c8m")):
    import torch

    import oclpathtracer_b200 as pt

    torch.cuda.init()
    stream = torch.cuda.current_stream()
    dev = pt.Device(0, stream=stream.cuda_stream)
    tris, mats = pt.load_model(os.path.join(ROOT, "data", "cornellbox.bin"))
    mats_t = torch.from_numpy(np.ascontiguousarray(mats).view(np.float32).reshape(-1, 16)).cuda()
    res = {"info": card_info(), "device": dev.name(), "reps": reps, "scenes": {}}

    def host_route(tris_t):
        t0 = time.perf_counter()
        h_tris = tris_t.cpu().numpy().view(pt.TRIANGLE_DTYPE).reshape(-1)
        h_mats = mats_t.cpu().numpy().view(pt.MATERIAL_DTYPE).reshape(-1)
        t1 = time.perf_counter()
        sc = dev.scene(h_tris, h_mats, gpu_build=True)
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        return sc, (t2 - t0) * 1e3, (t1 - t0) * 1e3, (t2 - t1) * 1e3

    def device_route(tris_t):
        t0 = time.perf_counter()
        sc = dev.scene_from_device(tris_t, mats_t)
        torch.cuda.synchronize()
        return sc, (time.perf_counter() - t0) * 1e3

    for name in only:
        big = pt.tessellate(tris, SCENES[name])
        tris_t = torch.from_numpy(np.ascontiguousarray(big).view(np.float32).reshape(-1, 16)).cuda()
        torch.cuda.synchronize()
        # warm-up, and the two scenes are the same scene
        a = host_route(tris_t)[0]
        b = device_route(tris_t)[0]
        assert a.info() == b.info(), (a.info(), b.info())
        na, oa = a.bvh()
        nb, ob_ = b.bvh()
        live = live_nodes(na)
        assert na[live].tobytes() == nb[live].tobytes() and oa.tobytes() == ob_.tobytes()
        frames = []
        prm = pt.default_params(width=3840, height=2160, n_frames=1, mode=pt.MODE_PATH, accum=pt.ACCUM_LINEAR, max_depth=8)
        for sc in (a, b):
            fb = dev.buffer(3840 * 2160 * 16)
            dev.render(sc, prm, fb)
            frames.append(fb.read(np.uint32).tobytes())
            fb.close()
        assert frames[0] == frames[1], name
        a.close(); b.close()
        host_ms, down_ms, create_ms, dev_ms = [], [], [], []
        for _ in range(reps):
            sc, t, td, tc = host_route(tris_t)
            sc.close()
            host_ms.append(t); down_ms.append(td); create_ms.append(tc)
            sc, t = device_route(tris_t)
            sc.close()
            dev_ms.append(t)
        # where the time goes: device time of every kernel and copy in one build of each route
        kernels = {}
        for route, fn in (("host", host_route), ("device", device_route)):
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CPU,
                                                    torch.profiler.ProfilerActivity.CUDA]) as prof:
                sc = fn(tris_t)[0]
            sc.close()
            rows = {}
            for ev in prof.key_averages():
                us = getattr(ev, "device_time_total", None)
                if us is None:
                    us = ev.cuda_time_total
                if us > 0:
                    rows[ev.key] = round(float(us) / 1e3, 4)
            kernels[route] = dict(sorted(rows.items(), key=lambda kv: -kv[1]))
        entry = {"triangles": len(big), "record_bytes": len(big) * 64, "c5_frame_bytes_identical": True,
                 "host_route_ms": host_ms, "host_download_ms": down_ms, "host_create_gpu_ms": create_ms, "device_route_ms": dev_ms,
                 "host_route_median_ms": float(np.median(host_ms)), "host_download_median_ms": float(np.median(down_ms)),
                 "host_create_gpu_median_ms": float(np.median(create_ms)), "device_route_median_ms": float(np.median(dev_ms)),
                 "speedup": float(np.median(host_ms) / np.median(dev_ms)), "device_time_ms": kernels}
        print(name, json.dumps({k: v for k, v in entry.items() if k != "device_time_ms"}), flush=True)
        res["scenes"][name] = entry
        del tris_t
        torch.cuda.empty_cache()
    dev.close()
    os.makedirs(out_dir, exist_ok=True)
    with open(os.path.join(out_dir, "bench_scene_build.json"), "w") as f:
        json.dump(res, f, indent=1)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--only", default="c5,c8m")
    a = ap.parse_args()
    res = run(a.out_dir, a.reps, tuple(a.only.split(",")))
    print(json.dumps(res["info"]))


if __name__ == "__main__":
    main()
