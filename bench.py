#!/usr/bin/env python
"""bench.py -- Mrays/s (primary + secondary) of the ray-cast + radiance path on B200.

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (through the C-ABI)
  python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on the host cores
  python bench.py ... --dump-outputs DIR                   # also writes the last timed step's image: compare two builds with it

Workload (default c5 = BASELINE.json configs[4], the configuration the metric is quoted on "at 1/2/4/8 GPUs"): the
2,005,056-triangle tessellated Cornell box, full path trace (max depth 8), 3840x2160, 64 spp.  One STEP = one pass of
the hot path over the WHOLE configuration: all 64 samples of every pixel of ONE image.  With N ranks the image is
tile-sharded (64-pixel blocks round-robin, strong scaling): each rank renders its tiles and the resolve kernel stores
every finished pixel into rank 0's image over NVLink peer memory (no collective on the data path), so a step ends with
ONE image.  value = rays of all ranks / sum over steps of the max-over-ranks device time.  configs[0..3] ride along as
sub-records (`configs`), each over its own full configuration.

Printed keys follow the driver's contract; see DESIGN.md "Measurement" for how each number is made.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
SCENE = os.path.join(ROOT, "data", "cornellbox.bin")

WORKLOADS = {
    # BASELINE.json configs[0..4]; spp = frames of one full pass over the configuration (= one step)
    "c1": dict(width=512, height=512, mode=0, spp=1, desc="cornellbox.bin primary-ray cast 512x512, 1 spp, hit-ID output"),
    "c2": dict(width=1024, height=1024, mode=1, ao_samples=16, spp=1, desc="cornellbox.bin ambient occlusion 1024x1024, 16 AO rays/pixel"),
    "c3": dict(width=1920, height=1080, mode=2, spp=64, desc="cornellbox.bin direct lighting with area-light shadow rays, 64 spp at 1920x1080"),
    "c4": dict(width=3840, height=2160, mode=3, max_depth=8, spp=256, desc="cornellbox.bin full path trace (max depth 8), 256 spp at 4K"),
    "c5": dict(width=3840, height=2160, mode=3, max_depth=8, tess=236, spp=64,
               desc="synthetic 2M-triangle tessellated scene (18 Cornell quads x 236^2 x 2 = 2,005,056 triangles), full path trace (max depth 8), 64 spp at 4K"),
}
METRIC = "Mrays/sec (primary+secondary)"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c5", choices=sorted(WORKLOADS))
    ap.add_argument("--spp-per-step", type=int, default=0, help="frames per step (0 = the configuration's full spp)")
    ap.add_argument("--integrator", default="auto", choices=["auto", "mega", "wavefront"])
    ap.add_argument("--accel", default="bvh", choices=["bvh", "brute"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-sub", action="store_true", help="skip the configs[0..3] sub-records")
    ap.add_argument("--tune", action="append", default=[], help="experiment knob index=value (ptb_device_set_tuning)")
    ap.add_argument("--fpb", type=int, default=0, help="frames_per_batch override")
    ap.add_argument("--smem-nodes", type=int, default=0, help="BVH nodes staged in shared memory (0 = default)")
    ap.add_argument("--max-leaf", type=int, default=0, help="BVH max triangles per leaf (0 = default)")
    ap.add_argument("--sah-traverse", type=float, default=0.0, help="SAH node-visit cost (0 = default 1.2)")
    ap.add_argument("--force-width", type=int, default=0, help="force the scene form: 1 FLAT, 4 4-wide, 2 binary (0 = the library's pick)")
    ap.add_argument("--gpu-build", action="store_true", help="build the BVH on the device (LBVH) instead of the host SAH builder")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the image of the last timed step to DIR/image.npy "
                                                          "(float32 RGBA rows; see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours (the reference arm times a shard whose size depends on the host)")
    return args


def dist_env():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))


def host_threads():
    """every CPU this process may run on -- NOT OMP_NUM_THREADS: torchrun exports OMP_NUM_THREADS=1 to its workers"""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def config_of(name, world):
    """`config` of the JSON line: the same dict for this repo's arm and for the reference arm"""
    wl = WORKLOADS[name]
    return {"workload": f"{name}: {wl['desc']}",
            "step": f"one full pass over the configuration: {wl['spp']} sample(s) per pixel of ONE {wl['width']}x{wl['height']} image",
            "scene_triangles": 36 * (wl.get("tess", 1) ** 2),
            "parallelism": f"image tile-sharded over {world} GPU(s) (64-pixel blocks round-robin), one image per step",
            "l2": "a 256 MiB flush runs between timed steps (and the 2M-triangle scene, 33 MB of quantised nodes + 96 MB of triangles, exceeds the 126 MB L2)"}


def bind_to_gpu_numa(gpu_index):
    """Pins this rank (and so its page-locked host buffers) to the CPUs next to its GPU; plumbing only, never fatal."""
    try:
        import pynvml
        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(gpu_index))
        return "numa-local (nvmlDeviceSetCpuAffinity), %d cpus" % len(os.sched_getaffinity(0))
    except Exception as e:
        return "unbound (%s)" % type(e).__name__


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,timestamp")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.gpu = [], None, gpu_index
        self.t0 = self.t1 = None

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def start(self):
        try:
            import shutil
            cmd = ["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50"]
            if shutil.which("stdbuf"):
                cmd = ["stdbuf", "-oL"] + cmd
            self.proc = subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except OSError:
            self.proc = None

    def _read(self):
        import datetime
        for line in self.proc.stdout:
            cols = [c.strip() for c in line.split(",")]
            ts = time.time()
            try:
                ts = datetime.datetime.strptime(cols[9], "%Y/%m/%d %H:%M:%S.%f").timestamp()
            except (IndexError, ValueError):
                pass
            self.rows.append((ts, cols))

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        lo, hi = (self.t0 or 0.0) - 0.03, (self.t1 or 1e18) + 0.03
        rows = [r for (ts, r) in self.rows if lo <= ts <= hi] or [r for (_, r) in self.rows[-3:]]

        def col(i):
            return [float(r[i]) for r in rows if len(r) >= 9 and r[i].replace(".", "").isdigit()]
        sm, mx, pw = col(1), col(2), col(3)
        reasons = set()
        for r in rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)", float(d.get("sm_max_mhz", 1965.0))
    return 6650.0, "fallback (B200_PROFILING.md)", 1965.0


DUMP_PIXELS = 1 << 21  # 32 MiB of float4 rows


def dump_outputs(path, image):
    """Writes `image` ((pixels, 4) float32, the image a caller of the timed path receives) as path/image.npy: whole when it has at most
    DUMP_PIXELS pixels, else the rows of DUMP_PIXELS pixels drawn once with seed 0 and kept in ascending order -- the same pixels on
    every run of the workload, so that the files of two builds compare row for row."""
    os.makedirs(path, exist_ok=True)
    if len(image) > DUMP_PIXELS:
        image = image[np.sort(np.random.default_rng(0).choice(len(image), DUMP_PIXELS, replace=False))]
    np.save(os.path.join(path, "image.npy"), np.ascontiguousarray(image, np.float32))


def ncu_traffic(name):
    """DRAM / L2 bytes of the dominant kernel from the committed `ncu --set full` capture (profiles/ncu_traffic.json)"""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    return (json.load(open(path)).get(name) or {}) if os.path.exists(path) else {}


# ------------------------------------------------------------------------------------------------------
# the oracle on the host cores: cpu_baseline of this repo's arm and the whole reference arm
# ------------------------------------------------------------------------------------------------------

class CpuPath:
    """The reference's algorithm restated on the CPU (oracle/: test infrastructure, the only CPU code bench.py runs).

    The reference has NO CPU executor of its own (ADL's DeviceHost cannot launch kernels, SURVEY.md section 0):
    oracle/_ref/adlTest64 is the genuine test program but it needs an OpenCL GPU platform (measured on the B200:
    profiles/reference_opencl_r02/), so kind = "port".  Cornell configurations run the reference's own brute-force loop
    over the 36 triangles (GenerateColors.cl:137-154).  The 2M-triangle scene cannot (72 G triangle tests per 4K frame):
    there the oracle walks its own BVH (oracle/oracle_bvh.c), stated in `algorithm`.
    """

    def __init__(self, name, n_threads=0, share=None):
        from oracle import binding as ob
        self.ob, self.name, self.wl = ob, name, WORKLOADS[name]
        self.n_threads = n_threads or host_threads()
        if share is not None:
            self.tris, self.mats, self.light, self.bvh, self.algorithm = share.tris, share.mats, share.light, share.bvh, share.algorithm
            return
        self.tris, self.mats = ob.load_model(SCENE)
        self.light = ob.light_from_quad(self.tris, 5)
        self.bvh = None
        if self.wl.get("tess"):
            self.tris = ob.tessellate(self.tris, self.wl["tess"])
            b = ob.build_bvh(self.tris)
            self.bvh, self._keep = ob.make_bvh(b["nodes"], b["tri_order"])
            self.algorithm = (f"the oracle's BVH path (its own binned-SAH tree over {len(self.tris)} triangles; the reference's brute-force loop "
                              "would be 72 G triangle tests per frame), OpenMP over pixels")
        else:
            self.algorithm = "reference brute-force loop over the 36 triangles (GenerateColors.cl:137-154) restated in C, OpenMP over pixels"

    def params(self, first_frame, n_frames, shard=None):
        wl, ob = self.wl, self.ob
        kw = dict(mode=wl["mode"], accum=ob.ACCUM_LINEAR, use_bvh=1 if self.bvh is not None else 0, light_p1=self.light[0],
                  light_ea=self.light[1], light_eb=self.light[2], n_threads=self.n_threads, first_frame=first_frame, n_frames=n_frames)
        if "ao_samples" in wl:
            kw["ao_samples"] = wl["ao_samples"]
        if "max_depth" in wl:
            kw["max_depth"] = wl["max_depth"]
        if shard:
            kw.update(shard_index=shard[0], shard_count=shard[1], shard_block=64)
        return ob.default_params(wl["width"], wl["height"], **kw)

    def sample(self, first_frame, shard_count):
        """one bounded sample: 1 spp of the 1/shard_count tile shard of the image that frame `first_frame` selects"""
        shard = (first_frame % shard_count, shard_count) if shard_count > 1 else None
        t0 = time.perf_counter()
        _, _, ctr = self.ob.render(self.params(first_frame, 1, shard), self.tris, self.mats, bvh=self.bvh)
        return ctr["rays_closest"] + ctr["rays_any"], time.perf_counter() - t0

    def calibrate(self, target_s):
        """shard count (a power of two) so that one sample takes about target_s on these cores"""
        self.sample(0, 64)             # cold: first touch of the tree
        _, secs = self.sample(1, 64)
        full, sc = secs * 64, 1
        while full / sc > target_s and sc < 4096:
            sc *= 2
        return sc

    def describe(self, shard_count, samples, rays, secs):
        wl = self.wl
        what = "the whole image" if shard_count == 1 else f"a 1/{shard_count} tile shard (64-pixel blocks) of the image"
        return f"{samples} sample(s) of 1 spp over {what} at {wl['width']}x{wl['height']} ({int(rays)} rays, {secs:.2f} s)"


def cpu_baseline(name, budget_s=12.0):
    cp = CpuPath(name)
    sc = cp.calibrate(1.5)
    rays = secs = n = 0
    while secs < budget_s and n < 64:
        r, s = cp.sample(n, sc)
        rays += r; secs += s; n += 1
    one = CpuPath(name, n_threads=1, share=cp)
    r1, s1 = one.sample(0, sc * 8)
    return {"value": rays / secs / 1e6, "unit": "Mrays/s", "cores": cp.n_threads, "kind": "port", "algorithm": cp.algorithm,
            "sample": cp.describe(sc, n, rays, secs),
            "single_thread": {"value": r1 / s1 / 1e6, "unit": "Mrays/s", "cores": 1}}


def run_reference_arm(args, rank, world):
    """--impl reference: the reference's algorithm on the host cores, same config / metric / unit as this repo's arm; each
    step is a bounded sample of the workload.  Under torchrun rank 0 alone runs and prints; the others exit 0."""
    if rank != 0:
        return
    cp = CpuPath(args.workload)
    sc = cp.calibrate(1.5)
    for i in range(args.warmup):
        cp.sample(i, sc)
    rays = secs = 0
    for i in range(args.steps):
        r, s = cp.sample(args.warmup + i, sc)
        rays += r; secs += s
    value = rays / secs / 1e6
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "Mrays/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": secs / max(1, args.steps) * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_of(args.workload, world),
        "cpu_baseline": {"value": value, "unit": "Mrays/s", "cores": cp.n_threads, "kind": "port", "algorithm": cp.algorithm,
                         "sample": "per step: " + cp.describe(sc, 1, rays / max(1, args.steps), secs / max(1, args.steps))},
        "e2e": {"value": value, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------
# this repo's arm
# ------------------------------------------------------------------------------------------------------

class Job:
    """One workload on this rank: resident scene, full images (double-buffered), rank 0's images mapped as peer memory."""

    def __init__(self, pt, dev, dist, rank, world, name, args, scene_cache):
        import torch
        self.pt, self.dev, self.dist, self.rank, self.world, self.name, self.args = pt, dev, dist, rank, world, name, args
        self.torch = torch
        self.wl = WORKLOADS[name]
        self.npix = self.wl["width"] * self.wl["height"]
        self.spp = args.spp_per_step if (args.spp_per_step and name == args.workload) else self.wl["spp"]
        key = self.wl.get("tess", 1)
        if key not in scene_cache:
            tris, mats = pt.load_model(SCENE)
            light = pt.light_from_quad(tris, 5)
            if self.wl.get("tess"):
                tris = pt.tessellate(tris, self.wl["tess"])
            bp = None
            if args.smem_nodes or args.max_leaf or args.sah_traverse or args.force_width:
                bp = pt.bvh_params()
                bp.force_width = args.force_width
                if args.sah_traverse:
                    bp.traverse_cost = args.sah_traverse
                if args.smem_nodes:
                    bp.smem_nodes = args.smem_nodes
                if args.max_leaf:
                    bp.max_leaf = args.max_leaf
            t0 = time.perf_counter()
            scene = dev.scene(tris, mats, bp, gpu_build=args.gpu_build)
            dev.sync()
            scene_cache[key] = (tris, mats, light, scene, time.perf_counter() - t0)
        self.tris, self.mats, self.light, self.scene, self.build_s = scene_cache[key]
        self.integ = {"auto": pt.INTEGRATOR_AUTO, "mega": pt.INTEGRATOR_MEGAKERNEL, "wavefront": pt.INTEGRATOR_WAVEFRONT}[args.integrator]
        self.accel = pt.ACCEL_BVH if args.accel == "bvh" else pt.ACCEL_BRUTE
        # every rank owns two full images; the two of rank 0 are mapped into the other ranks (CUDA IPC over NVLink)
        self.full = [dev.buffer(self.npix * 16) for _ in range(2)]
        for b in self.full:
            b.clear()
        dev.sync()
        self.peer = [[], []]
        self.imported = []
        if world > 1:
            handles = [[b.ipc_export() for b in self.full]] if rank == 0 else [None]
            dist.broadcast_object_list(handles, src=0)
            if rank != 0:
                self.imported = [dev.ipc_import(h, self.npix * 16) for h in handles[0]]
                self.peer = [[self.imported[0]], [self.imported[1]]]

    def params(self, i, **kw):
        pt, wl = self.pt, self.wl
        p = pt.default_params(width=wl["width"], height=wl["height"], mode=wl["mode"], accum=pt.ACCUM_LINEAR, first_frame=i * self.spp,
                              n_frames=self.spp, integrator=self.integ, accel=self.accel, frames_per_batch=self.args.fpb,
                              shard_index=self.rank, shard_count=self.world, shard_block=64, **kw)
        if "ao_samples" in wl:
            p.ao_samples = wl["ao_samples"]
        if "max_depth" in wl:
            p.max_depth = wl["max_depth"]
        p.light_p1[:], p.light_ea[:], p.light_eb[:] = self.light
        return p

    def step(self, i, which=0):
        """one pass of the hot path over the configuration: this rank's tiles, delivered into rank 0's image by the resolve kernel"""
        self.dev.render_gather(self.scene, self.params(i), self.full[which], self.peer[which])

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def reduce(self, values, op):
        t = self.torch.tensor(values, dtype=self.torch.float64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t, op={"max": self.dist.ReduceOp.MAX, "sum": self.dist.ReduceOp.SUM}[op])
        return [float(x) for x in t]

    def device_timed(self, steps, warmup, flush, stream, sampler=None):
        """(rays of all ranks, total ms = sum over steps of the max-over-ranks device time, per-step ms, profile)"""
        torch, dev = self.torch, self.dev
        for i in range(warmup):
            self.step(i)
        self.barrier()
        dev.counters(cumulative=1, read=False)
        dev.profile(True)
        dev.profile_read()
        if sampler:
            sampler.mark_begin()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for i in range(steps):
            flush.fill_(i & 255)           # evict L2 between timed iterations (untimed)
            ev[i][0].record(stream)
            self.step(warmup + i)
            ev[i][1].record(stream)
        self.barrier()
        if sampler:
            sampler.mark_end()
        prof = dev.profile_read()
        dev.profile(False)
        ctr = dev.counters(cumulative=0, read=True)
        ms = self.reduce([a.elapsed_time(b) for a, b in ev], "max")
        rays = self.reduce([ctr["rays_closest"] + ctr["rays_any"]], "sum")[0]
        return rays, sum(ms), ms, prof

    def e2e(self, steps, rgb8=False):
        """The same metric end to end through the C-ABI with HOST buffers, per step and per rank: H2D of the caller's scene records
        from page-locked memory (ptb_buffer_write, on an upload queue of its own: the render reads the resident scene built
        from identical records), ptb_render_gather of this rank's tiles into rank 0's image, a barrier, and on rank 0 the D2H
        of the ONE finished image into page-locked host memory (ptb_buffer_read on a copy queue; the copy of step i overlaps
        the render of step i+1: two images alternate).  Host wall clock, max over ranks."""
        pt, dev, torch = self.pt, self.dev, self.torch
        up = pt.Device(torch.cuda.current_device())   # upload queue
        cp = pt.Device(torch.cuda.current_device())   # read-back queue (rank 0)
        tp, mp = pt.PinnedArray(self.tris.shape, self.tris.dtype), pt.PinnedArray(self.mats.shape, self.mats.dtype)
        tp.array[...] = self.tris
        mp.array[...] = self.mats
        rec_t, rec_m = up.buffer(self.tris.nbytes), up.buffer(self.mats.nbytes)
        outs, views, rgbs = [], [], []
        if self.rank == 0:
            for k in range(2):
                if rgb8:
                    rgbs.append(dev.buffer((self.npix * 3 + 15) // 16 * 16))
                    views.append(cp.wrap(rgbs[k].device_ptr(), self.npix * 3))
                    outs.append(pt.PinnedArray((self.npix, 3), np.uint8))
                else:
                    views.append(cp.wrap(self.full[k].device_ptr(), self.npix * 16))
                    outs.append(pt.PinnedArray((self.npix, 4), np.float32))

        def loop(n):
            t0 = time.perf_counter()
            for i in range(n):
                w = i & 1
                rec_t.write_async(tp.array)            # H2D: this step's inputs
                rec_m.write_async(mp.array)
                self.step(i, w)                        # render + fused gather into rank 0's image w
                if self.rank == 0:
                    cp.sync()                          # image w^1 (step i-1) has reached the host while step i rendered
                dev.sync()
                up.sync()
                if self.world > 1:
                    self.dist.barrier()                # every rank's tiles are in rank 0's image
                    torch.cuda.synchronize()
                if self.rank == 0:
                    if rgb8:
                        self.full[w].to_rgb8(self.npix, rgbs[w])
                        dev.sync()
                    views[w].read_async(outs[w].array)  # D2H of the ONE image
            if self.rank == 0:
                cp.sync()
            return time.perf_counter() - t0

        loop(2)
        self.barrier()
        dev.counters(cumulative=1, read=False)
        t = loop(steps)
        ctr = dev.counters(cumulative=0, read=True)
        self.barrier()
        checksum = float(outs[(steps - 1) & 1].array[::4097].astype(np.float64).sum()) if self.rank == 0 else 0.0
        t_max = self.reduce([t], "max")[0]
        rays = self.reduce([ctr["rays_closest"] + ctr["rays_any"]], "sum")[0]
        for b in views + rgbs + [rec_t, rec_m]:
            b.close()
        for pa in [tp, mp] + outs:
            pa.free()
        up.close(); cp.close()
        return {"value": rays / t_max / 1e6, "unit": "Mrays/s", "ms_per_step": t_max / steps * 1e3,
                "h2d_bytes_per_step": int((self.tris.nbytes + self.mats.nbytes) * self.world),
                "d2h_bytes_per_step": int(self.npix * (3 if rgb8 else 16)), "host_checksum": checksum, "steps": steps}

    def image(self):
        """rank 0's image of the last device_timed step, (pixels, 4) float32"""
        return self.full[0].read(np.float32).reshape(-1, 4)

    def close(self):
        self.barrier()
        for b in self.imported:
            b.close()
        self.barrier()
        for b in self.full:
            b.close()


def simt_fraction(job, rays_per_s, sm_count, sm_max_mhz):
    """fp32 lane-ops of traversal per ray (SURVEY.md 8d: slab 24 per box, Moller-Trumbore stages 14/10/15/6/40) from the oracle's exact
    stage counts on a reduced image of the same configuration, times the measured ray rate, over the no-FMA issue peak."""
    from oracle import binding as ob
    wl = job.wl
    otris, omats = ob.load_model(SCENE)
    p1, ea, eb = ob.light_from_quad(otris, 5)
    if wl.get("tess"):
        otris = ob.tessellate(otris, wl["tess"])
    width = job.scene.mode_width(wl["mode"])
    b = ob.build_bvh(otris, width=width)
    bvh, _keep = ob.make_bvh(b["nodes"], b["tri_order"])
    kw = dict(n_frames=1, mode=wl["mode"], accum=1, use_bvh=1, ao_samples=wl.get("ao_samples", 16), max_depth=wl.get("max_depth", 16),
              light_p1=p1, light_ea=ea, light_eb=eb, n_threads=host_threads())
    if wl.get("tess"):
        op = ob.default_params(wl["width"], wl["height"], shard_index=7, shard_count=64, shard_block=64, **kw)
    else:
        op = ob.default_params(256, 256, **kw)
    _, _, oc = ob.render(op, otris, omats, bvh=bvh)
    nr = oc["rays_closest"] + oc["rays_any"]
    boxes = nr * len(b["nodes"]) if width == 1 else oc["nodes"] * width  # FLAT: every leaf box for every ray
    flops = (boxes * 24 + oc["tri_tests"] * 14 + oc["tri_u"] * 10 + oc["tri_v"] * 15 + oc["tri_t"] * 6 + oc["tri_accept"] * 40) / nr
    peak = sm_count * 128 * sm_max_mhz * 1e6  # no FMA in the parity build: one lane-op per lane per clock
    return {"bound": "fp32_issue", "flops_per_ray": flops, "boxes_per_ray": boxes / nr, "nodes_per_ray": oc["nodes"] / nr,
            "tri_tests_per_ray": oc["tri_tests"] / nr, "achieved_tlaneops": flops * rays_per_s / 1e12, "peak_tlaneops": peak / 1e12,
            "frac": flops * rays_per_s / peak,
            "scene_form": {1: "FLAT (every leaf box, no tree)", 4: "4-wide tree", 2: "binary tree"}.get(width, str(width)),
            "note": "algorithmic fp32 ops of traversal only; shading, RNG and sin/cos are extra"}


def main():
    sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree, __pycache__ included
    args = parse()
    rank, world, local = dist_env()
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    import oclpathtracer_b200 as pt

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU path (use --impl reference for the host baseline)")
    torch.cuda.set_device(local)
    affinity = bind_to_gpu_numa(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    stream = torch.cuda.current_stream()
    dev = pt.Device(local, stream=stream.cuda_stream)  # enqueue on torch's stream so torch events see the work
    for kv in args.tune:
        i, v = kv.split("=")
        dev.set_tuning(int(i), int(v))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")       # > 126 MB L2
    hbm_peak, peak_src, sm_max_mhz = peaks()
    sm_count = dev.sm_count()
    scenes = {}

    # ---- the workload the metric is quoted on ------------------------------------------------------------------
    job = Job(pt, dev, dist, rank, world, args.workload, args, scenes)
    sampler = ClockSampler(local)
    sampler.start()
    try:
        rays_all, ms_total, ms_steps, prof = job.device_timed(args.steps, args.warmup, flush, stream, sampler)
    finally:
        clocks = sampler.stop()  # no nvidia-smi left running if the timed steps fail
    if args.dump_outputs:
        if rank == 0:
            dump_outputs(args.dump_outputs, job.image())
        job.barrier()  # e2e() on every rank renders into rank 0's images
    value = rays_all / (ms_total * 1e-3) / 1e6
    launches = int(prof["kernel_launches"])
    e2e = None
    if not args.no_e2e:
        ne = max(2, min(args.steps, 5))
        e2e = job.e2e(ne)
        e2e["rgb8"] = {k: v for k, v in job.e2e(ne, rgb8=True).items() if k in ("value", "unit", "ms_per_step", "d2h_bytes_per_step")}
        e2e["timing"] = ("host wall clock over the steps, max over ranks; per step and rank: ptb_buffer_write of the scene records from page-locked "
                         "memory (H2D), ptb_render_gather of the rank's tiles into rank 0's image, barrier, rank 0 reads the ONE float4 image "
                         "back into page-locked memory (ptb_buffer_read; overlaps the next step's render).  rgb8: the image travels as the "
                         "reference's 8-bit output (RaytraceTest.cpp:78-83,:283 run on the device), 3 bytes per pixel")

    # ---- roofline of the dominant kernel --------------------------------------------------------------------------
    wl = job.wl
    integ_ms = prof["integrator_ms"] / max(1, prof["batches"])          # mean duration of one integrator launch (CUDA events, live)
    rays_per_launch = rays_all / world / max(1, prof["batches"])
    tr = ncu_traffic(args.workload)
    roof = {"kernel": ("k_path_sm2" if wl.get("tess") else "k_mega_path_regen") if wl["mode"] == 3 else "k_mega", "kernel_ms": integ_ms,
            "launches_per_step": prof["batches"] / max(1, args.steps),
            "kernel_share_of_step": (prof["integrator_ms"] / max(1e-9, sum(ms_steps))) if world == 1 else None,
            "rays_per_launch": rays_per_launch, "peak_source": peak_src}
    simt = simt_fraction(job, rays_per_launch / (integ_ms * 1e-3), sm_count, sm_max_mhz) if rank == 0 else None
    if rank == 0 and wl.get("tess"):
        # Scene traversed from L2/HBM.  Four lines, all <= 1 (profiles/ncu_traffic.json holds the per-ray counts of the committed
        # `ncu --set full` capture of this kernel; the rate is measured live with CUDA events):
        #   top level = issue slots: warp instructions per ray x rays/s against one instruction per clock and scheduler -- the unit
        #               closest to saturation since the nodes are 32-byte records (before, the L1 data pipe was, at 84 %);
        #   l1        = the L1 data pipe: L1 wavefronts per ray (one per lane and node visit) against one per clock and SM;
        #   hbm       = the contract's HBM line from the DRAM bytes ncu measured (the tree's cold levels and the triangles);
        #   l2        = SURVEY 8d's algorithmic bytes per ray (nodes*32 + tri_tests*48 + 16 B/sample: the L1/L2 stream) against the L2 cap.
        alg = simt["nodes_per_ray"] * 32 + simt["tri_tests_per_ray"] * 48 + 16.0 * job.npix * job.spp / max(1.0, rays_all / args.steps)
        dram = tr.get("dram_bytes_per_ray")
        wpr = tr.get("l1_wavefronts_per_ray")
        ipr = tr.get("warp_instructions_per_ray")
        rate = rays_per_launch / (integ_ms * 1e-3)
        l2_peak = 6300.0 * sm_max_mhz * 1e6 / 1e9  # LTS cap ~6300 B/clk (B300_MICROARCH.md; same L2 design) at this GPU's clock
        l1_peak = sm_count * sm_max_mhz * 1e6 / 1e9  # G wavefronts/s: one per clock and SM
        issue_peak = 4 * sm_count * sm_max_mhz * 1e6 / 1e9  # G warp instructions/s: one per clock and scheduler
        roof.update({"bound": "issue_slots", "achieved": ipr * rate / 1e9 if ipr else None, "peak": issue_peak, "unit": "G warp-inst/s",
                     "frac": ipr * rate / 1e9 / issue_peak if ipr else None, "traffic": dram * rays_per_launch if dram else None,
                     "warp_instructions_per_ray": ipr, "active_lanes_per_instruction": (tr.get("ncu") or {}).get("active_lanes_per_instruction"),
                     "ncu": tr.get("ncu"),
                     "l1": {"achieved": wpr * rate / 1e9 if wpr else None, "peak": l1_peak, "unit": "G wavefront/s",
                            "frac": wpr * rate / 1e9 / l1_peak if wpr else None, "l1_wavefronts_per_ray": wpr},
                     "hbm": {"achieved": dram * rate / 1e9 if dram else None, "peak": hbm_peak, "unit": "GB/s", "frac": dram * rate / 1e9 / hbm_peak if dram else None,
                             "dram_bytes_per_ray": dram},
                     "l2": {"algorithmic_bytes_per_ray": alg, "achieved": alg * rate / 1e9, "peak": l2_peak, "unit": "GB/s", "frac": alg * rate / 1e9 / l2_peak,
                            "note": "SURVEY 8d's algorithmic bytes (nodes*32 [quantised 32-byte records] + tri_tests*48 + 16 B/sample) are the L1/L2 stream, quoted against the L2 bandwidth cap"},
                     "simt": simt,
                     "binding": "issue slots (ncu: 73 % busy at 15.2 of 32 lanes) and the L1 data pipe (74 %) together with long-scoreboard stalls on dependent "
                                "node fetches (7.5 per issue, 12 CTAs of 4 warps per SM); L2 at 40 %, HBM at 9 %",
                     "note": "achieved = warp instructions per ray of the committed ncu capture (profiles/ncu_traffic.json) x rays per second measured live with CUDA "
                             "events; traffic = dram__bytes_read + dram__bytes_write per launch of the same capture scaled to this launch's rays"})
    elif rank == 0:
        roof.update({"bound": "fp32_issue", "achieved": simt["achieved_tlaneops"], "peak": simt["peak_tlaneops"], "unit": "T lane-op/s",
                     "frac": simt["frac"], "traffic": tr.get("dram_bytes_per_launch"), "simt": simt,
                     "note": "the 5 KB scene is shared-memory resident: HBM sees only the 16 B/sample radiance stream; the binding limit is fp32 issue (SURVEY 8d)"})

    # ---- configs[0..3] as sub-records ---------------------------------------------------------------------------------
    subs = {}
    if not args.no_sub:
        for name in ("c1", "c2", "c3", "c4"):
            if name == args.workload:
                continue
            sj = Job(pt, dev, dist, rank, world, name, args, scenes)
            sj.step(0); sj.barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream); sj.step(1); b.record(stream); sj.barrier()
            one_ms = sj.reduce([a.elapsed_time(b)], "max")[0]
            reps = int(min(2000, max(3, 250.0 / max(one_ms, 1e-3))))   # >= 0.25 s of timed steps
            r_all, ms_tot, _, sprof = sj.device_timed(reps, 3, flush, stream)
            cfg = config_of(name, world)
            rec = {"workload": cfg["workload"], "step": cfg["step"], "value": r_all / (ms_tot * 1e-3) / 1e6, "unit": "Mrays/s",
                   "ms_per_step": ms_tot / reps, "steps": reps, "spp_per_s": reps * sj.spp / (ms_tot * 1e-3)}
            if rank == 0:
                s_ms = sprof["integrator_ms"] / max(1, sprof["batches"])
                rec["simt"] = simt_fraction(sj, (r_all / world / max(1, sprof["batches"])) / (s_ms * 1e-3), sm_count, sm_max_mhz)
                rec["simt_frac"] = rec["simt"]["frac"]
            if not args.no_e2e:
                e = sj.e2e(int(min(300, max(3, 150.0 / max(one_ms, 1e-3)))))
                rec["e2e"] = {k: e[k] for k in ("value", "unit", "ms_per_step", "h2d_bytes_per_step", "d2h_bytes_per_step", "steps")}
            subs[name] = rec
            sj.close()

    # ---- CPU baseline beside it (rank 0, N=1 only) ------------------------------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline(args.workload)
        ref = os.path.join(ROOT, "profiles", "reference_opencl_r02", "timing.json")
        if os.path.exists(ref):  # recorded once, not re-measured here: the unmodified reference on this GPU through OpenCL
            cpu["reference_opencl_on_b200"] = json.load(open(ref))

    if rank == 0:
        cfg = config_of(args.workload, world)
        if job.spp != wl["spp"]:
            cfg["step"] = f"{job.spp} sample(s) per pixel of ONE {wl['width']}x{wl['height']} image (--spp-per-step)"
        line = {
            "metric": METRIC, "value": value, "unit": "Mrays/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_total / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": cfg,
            "details": {"integrator": args.integrator, "accel": args.accel, "scene_form": job.scene.info()["width"], "cpu_affinity": affinity,
                        "rays_per_step": rays_all / args.steps, "bvh_build_s": job.build_s, "sm_count": sm_count,
                        "exchange": "fused into the resolve kernel: 16-byte stores into rank 0's image over NVLink peer memory; a barrier ends the step",
                        "timing": "CUDA events per step on the launching stream; per step the MAX over ranks, summed over the steps"},
            "spp_per_s": args.steps * job.spp / (ms_total * 1e-3), "msamples_per_s": job.npix * job.spp * args.steps / (ms_total * 1e-3) / 1e6,
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches,
            "roofline": roof, "cpu_baseline": cpu, "configs": subs,
        }
        print(json.dumps(line), flush=True)
    job.close()
    for _, _, _, scene, _ in scenes.values():
        scene.close()
    dev.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
