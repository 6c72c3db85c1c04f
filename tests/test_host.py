"""CPU tests of the product's host side: C-ABI surface, loader, BVH builder, sharding, error paths."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from conftest import ROOT, SCENE


def test_library_exports_every_declared_symbol(pt):
    hdr = open(os.path.join(ROOT, "include", "ptb200.h")).read()
    declared = sorted(set(re.findall(r"\b(ptb_[a-z0-9_]+)\s*\(", hdr)))
    assert len(declared) >= 40
    lib = pt.lib()
    missing = [s for s in declared if not hasattr(lib, s)]
    assert not missing, missing
    assert sorted(pt.EXPORTS) == declared
    assert lib.ptb_version() == 100


def test_struct_sizes_match_reference_layout(pt):
    # RaytraceTest.cpp:50-76 / GenerateColors.cl:12-28: 64-byte packed records
    assert pt.TRIANGLE_DTYPE.itemsize == 64 and pt.MATERIAL_DTYPE.itemsize == 64
    assert pt.TRIANGLE_DTYPE.fields["id"][1] == 48
    assert pt.MATERIAL_DTYPE.fields["roughness"][1] == 32 and pt.MATERIAL_DTYPE.fields["type"][1] == 36
    assert pt.NODE_DTYPE.itemsize == 64 and pt.NODE4_DTYPE.itemsize == 128 and pt.BVH_TRI_DTYPE.itemsize == 48 and pt.STATS_DTYPE.itemsize == 32
    assert C.sizeof(pt.RenderParams) % 4 == 0 and C.sizeof(pt.Counters) == 64


def test_loader_matches_oracle_bytes(pt, ob):
    t1, m1 = pt.load_model(SCENE)
    t2, m2 = ob.load_model(SCENE)
    assert t1.tobytes() == t2.tobytes() and m1.tobytes() == m2.tobytes()


def test_loader_errors(pt, tmp_path):
    with pytest.raises(pt.PtbError, match="cannot open"):
        pt.load_model(str(tmp_path / "missing.bin"))
    bad = tmp_path / "bad.bin"
    bad.write_bytes(open(SCENE, "rb").read()[:700])
    with pytest.raises(pt.PtbError, match="truncated"):
        pt.load_model(str(bad))
    empty = tmp_path / "empty.bin"
    empty.write_bytes(b"")
    with pytest.raises(pt.PtbError):
        pt.load_model(str(empty))


def _validate_bvh(pt, tris, b, pad_min=0.0):
    nodes, order, otris = b["nodes"], b["tri_order"], b["ordered_tris"]
    n = len(tris)
    assert sorted(order.tolist()) == list(range(n))  # every triangle in exactly one leaf slot
    np.testing.assert_array_equal(otris["index"], order)
    np.testing.assert_array_equal(otris["quad"], tris["id"][order])
    np.testing.assert_array_equal(otris["p1"], tris["p1"][order][:, :3])
    np.testing.assert_array_equal(otris["e1"], (tris["p2"][order] - tris["p1"][order])[:, :3])  # GenerateColors.cl:92
    np.testing.assert_array_equal(otris["e2"], (tris["p3"][order] - tris["p1"][order])[:, :3])  # GenerateColors.cl:93
    tri_lo = np.minimum(np.minimum(tris["p1"], tris["p2"]), tris["p3"])[:, :3]
    tri_hi = np.maximum(np.maximum(tris["p1"], tris["p2"]), tris["p3"])[:, :3]
    covered = np.zeros(n, bool)
    seen_nodes = np.zeros(len(nodes), bool)

    def bounds(ref):
        """returns (lo, hi) of the subtree; checks containment recursively (iteratively for depth safety)"""
        if ref < 0:
            code = (~ref) & 0xFFFFFFFF
            first, count = code >> 3, (code & 7) + 1
            assert 1 <= count <= 8 and first + count <= n
            assert not covered[first:first + count].any()
            covered[first:first + count] = True
            idx = order[first:first + count]
            assert (np.diff(idx) > 0).all() if count > 1 else True  # ascending caller index inside a leaf
            return tri_lo[idx].min(0), tri_hi[idx].max(0)
        assert not seen_nodes[ref]
        seen_nodes[ref] = True
        nd = nodes[ref]
        lo_all, hi_all, used = [], [], 0
        for k in range(b["width"]):  # box k = [c_k - e_k, c_k + e_k]
            ch = int(nd[f"child{k}"])
            c, e = nd[f"c{k}"].astype(np.float64), nd[f"e{k}"].astype(np.float64)
            if ch == 0x7FFFFFFF:
                assert (e < 0).all()  # unused slot: can never be hit
                continue
            used += 1
            l, h = bounds(ch)
            assert (e > 0).all() and (c - e <= l - pad_min).all() and (c + e >= h + pad_min).all()
            lo_all.append(l); hi_all.append(h)
        assert used >= 2
        return np.minimum.reduce(lo_all), np.maximum.reduce(hi_all)

    import sys
    sys.setrecursionlimit(10000)
    bounds(0)
    assert covered.all() and seen_nodes.all()


@pytest.mark.parametrize("k,kw", [(1, {}), (4, {}), (4, {"max_leaf": 2, "smem_nodes": 64}), (12, {}), (12, {"traverse_cost": 2.5, "n_bins": 8}), (236, {})])
def test_product_tree_equals_oracle_tree(pt, ob, cornell, k, kw):
    """The oracle has its own deterministic builder (oracle/oracle_bvh.c, rules R1-R7); the product's host builder
    (csrc/bvh_build.cpp) must produce the same bytes in every form the scene qualifies for -- node-visit parity then does
    not lean on the product's own tree (SURVEY.md 7.1 step 6).  k = 236 is the 2,005,056-triangle scene of configs[4]."""
    tris, _ = cornell
    scene = tris if k == 1 else pt.tessellate(tris, k)
    widths = [2] + ([4] if len(scene) <= 2048 else []) + ([1] if len(scene) <= 64 else [])
    for width in widths:
        o = ob.build_bvh(scene, ob.bvh_params(**kw) if kw else None, width=width)
        p = pt.build_bvh_host(scene, pt.bvh_params(**kw) if kw else None, width=width)
        assert p["nodes"].view(np.uint8).tobytes() == o["nodes"].view(np.uint8).tobytes(), (k, width)
        assert np.array_equal(p["tri_order"], o["tri_order"]) and p["depth"] == o["depth"] and p["smem_nodes"] == o["bfs_nodes"]


def test_flat_form_of_tiny_scenes(pt, ob, cornell):
    """FLAT form (<= 32 leaves, <= 64 triangles): one record per leaf in leaf order, masks partition the triangle positions."""
    tris, _ = cornell
    b = pt.build_bvh_host(tris)
    assert b["width"] == 1 and len(b["nodes"]) == 18 and b["depth"] == 1
    m = b["nodes"]["mask_lo"].astype(np.uint64) | (b["nodes"]["mask_hi"].astype(np.uint64) << np.uint64(32))
    assert int(np.bitwise_or.reduce(m)) == (1 << 36) - 1 and sum(bin(int(x)).count("1") for x in m) == 36
    assert all(int(m[i]) < int(m[i + 1]) for i in range(len(m) - 1))  # leaf order == triangle order
    b2 = pt.build_bvh_host(tris, width=2)
    for i, rec in enumerate(b["nodes"]):  # every leaf box contains its triangles (padded)
        pos = [k for k in range(36) if (int(m[i]) >> k) & 1]
        v = np.concatenate([np.stack([tris[n][b["tri_order"][pos]][:, :3] for n in ("p1", "p2", "p3")])])
        assert (v.reshape(-1, 3) >= rec["c"] - rec["e"]).all() and (v.reshape(-1, 3) <= rec["c"] + rec["e"]).all()
    np.testing.assert_array_equal(b2["tri_order"], b["tri_order"])
    with pytest.raises(pt.PtbError, match="FLAT"):
        pt.build_bvh_host(pt.tessellate(tris, 2), width=1)
    one = pt.build_bvh_host(tris[:1], width=1)
    assert len(one["nodes"]) == 1 and one["nodes"]["mask_lo"][0] == 1


def test_bvh_structure_cornell(pt, cornell):
    tris, _ = cornell
    b = pt.build_bvh_host(tris, width=4)
    assert b["width"] == 4 and b["smem_nodes"] == len(b["nodes"]) <= 17 and 1 <= b["depth"] <= 8
    _validate_bvh(pt, tris, b, pad_min=5e-4)  # default pad = 1e-4 * diagonal(9.6) ~ 9.6e-4
    b2 = pt.build_bvh_host(tris, width=2)
    assert b2["smem_nodes"] == len(b2["nodes"]) <= 35 and 1 <= b2["depth"] <= 12
    np.testing.assert_array_equal(b2["tri_order"], b["tri_order"])  # same tree, collapsed
    _validate_bvh(pt, tris, b2, pad_min=5e-4)


@pytest.mark.parametrize("k,max_leaf,width", [(4, 4, 2), (4, 4, 4), (12, 2, 2), (9, 8, 2), (7, 3, 4)])
def test_bvh_structure_tessellated(pt, cornell, k, max_leaf, width):
    tris, _ = cornell
    big = pt.tessellate(tris, k)
    b = pt.build_bvh_host(big, pt.bvh_params(max_leaf=max_leaf, smem_nodes=64), width=width)
    assert b["smem_nodes"] == min(64, len(b["nodes"]))
    _validate_bvh(pt, big, b, pad_min=5e-4)
    # breadth-first prefix: children of early nodes come later, prefix is closed under "parent of"
    kids = np.concatenate([b["nodes"][f"child{k}"] for k in range(width)])
    assert (kids[(kids >= 0) & (kids != 0x7FFFFFFF)] > 0).all()


def test_bvh_degenerate_inputs(pt, cornell):
    tris, _ = cornell
    one = pt.build_bvh_host(tris[:1], width=4)
    assert len(one["nodes"]) == 1 and one["nodes"]["child0"][0] == one["nodes"]["child1"][0] < 0
    assert one["nodes"]["child2"][0] == one["nodes"]["child3"][0] == 0x7FFFFFFF
    same = np.repeat(tris[:1], 9)  # identical centroids: no bin separates them -> median split fallback
    for width in (2, 4):
        _validate_bvh(pt, same, pt.build_bvh_host(same, width=width))
    with pytest.raises(pt.PtbError, match="2048"):
        pt.build_bvh_host(pt.tessellate(tris, 12), width=4)
    bad = tris[:2].copy()
    bad["p1"][0, 0] = np.nan
    with pytest.raises(pt.PtbError, match="non-finite"):
        pt.build_bvh_host(bad)


def test_light_and_tessellate_helpers(pt, ob, cornell):
    tris, _ = cornell
    assert pt.light_from_quad(tris, 5) == ob.light_from_quad(tris, 5)
    p1, ea, eb = pt.light_from_quad(tris, 5)
    area = np.linalg.norm(np.cross(ea, eb))
    assert abs(area - 1.365) < 1e-3  # SURVEY App. B: light area 1.365
    assert np.cross(ea, eb)[1] < 0  # front side faces -y (into the room)
    with pytest.raises(pt.PtbError):
        pt.light_from_quad(tris, 99)
    with pytest.raises(pt.PtbError):
        pt.tessellate(tris[:3], 2)


def test_ppm_writer(pt, ob, tmp_path):
    # RaytraceTest.cpp:277-287: "P3\n%d %d\n%d\n" + "%d %d %d " per pixel, value = min((int)(sqrtf(v)*255),255)
    rng = np.random.default_rng(0)
    fb = rng.uniform(0, 1.5, (6, 4)).astype(np.float32)
    path = tmp_path / "out.ppm"
    pt.write_ppm(str(path), fb, 3, 2)
    txt = path.read_text()
    assert txt.startswith("P3\n3 2\n255\n")
    vals = [int(v) for v in txt.split()[4:]]
    assert vals == ob.to_rgb8(fb).reshape(-1).tolist() == pt.to_rgb8(fb).reshape(-1).tolist()


def test_no_cpu_fallback_without_gpu(pt):
    """On a box without CUDA the product refuses to run (no silent CPU path)."""
    n = C.c_int(-1)
    rc = pt.lib().ptb_device_count(C.byref(n))
    if rc == 0 and n.value > 0:
        pytest.skip("a CUDA device is present")
    with pytest.raises(pt.PtbError, match="no CUDA device|no CPU fallback"):
        pt.Device(0)


def test_render_params_defaults_equal_reference_constants(pt):
    p = pt.default_params()
    assert (p.width, p.height) == (512, 512)  # RaytraceTest.cpp:219
    assert p.max_depth == 16  # GenerateColors.cl:5 BOUNCES
    assert p.accum == pt.ACCUM_REFERENCE and p.mode == pt.MODE_PATH
    assert p.light_quad == 5 and p.shard_count == 1
    assert pt.local_pixels(p) == 512 * 512
    q = pt.default_params(width=40, height=25, shard_index=1, shard_count=3, shard_block=64)
    from oclpathtracer_b200 import sharding
    assert pt.local_pixels(q) == sharding.local_pixels(1000, 1, 3, 64) == 320


def test_product_never_imports_oracle():
    """The oracle is test infrastructure: no product source may reference it."""
    pkg = os.path.join(ROOT, "oclpathtracer_b200")
    for base, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                src = open(os.path.join(base, f), errors="ignore").read()
                for needle in ("oracle_pt", "liboracle", "from oracle", "import oracle", "oracle/"):
                    assert needle not in src, (f, needle)
    for f in os.listdir(os.path.join(ROOT, "include")):
        src = open(os.path.join(ROOT, "include", f)).read()
        for needle in ("oracle_pt", "liboracle", "oracle/"):
            assert needle not in src, (f, needle)


def test_raycast_host_program_refuses_without_gpu(pt, tmp_path):
    """The C++ mirror of DeviceTest.RayCast (host/raycast_main.cpp) exits loudly when there is no device."""
    import subprocess
    exe = os.path.join(ROOT, "oclpathtracer_b200", "host", "ptb_raycast")
    if not os.path.exists(exe):
        subprocess.check_call(["make", "-s", "-C", os.path.dirname(exe)])
    n = C.c_int(-1)
    if pt.lib().ptb_device_count(C.byref(n)) == 0 and n.value > 0:
        pytest.skip("a CUDA device is present")
    r = subprocess.run([exe, SCENE, str(tmp_path / "unused.ppm"), "32", "1"], capture_output=True, text=True)
    assert r.returncode == 2 and "no CUDA device" in r.stderr


def _gloo_worker(rank, world, port, w, h, block, q):
    import torch
    import torch.distributed as dist
    from oracle import binding as ob
    from oclpathtracer_b200 import sharding

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    tris, mats = ob.load_model(SCENE)
    # each rank renders its shard (the oracle stands in for the GPU renderer on this CPU-only box)
    prm = ob.default_params(w, h, n_frames=2, mode=3, accum=1, max_depth=4, shard_index=rank, shard_count=world,
                            shard_block=block, n_threads=2)
    local, _, _ = ob.render(prm, tris, mats)
    assert local.shape[0] == sharding.local_pixels(w * h, rank, world, block)
    img = sharding.gather_image(torch.from_numpy(local), w * h, rank, world, block)
    # frame sharding (bench.py's weak-scaling path): reduce(sum) of per-rank linear accumulators
    fr = ob.default_params(w, h, first_frame=rank, n_frames=1, mode=3, accum=1, max_depth=4, n_threads=2)
    mine, _, _ = ob.render(fr, tris, mats)
    acc = torch.from_numpy(mine.copy())
    dist.reduce(acc, dst=0, op=dist.ReduceOp.SUM)
    if rank == 0:
        q.put((img.numpy().tobytes(), acc.numpy().tobytes()))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("w,h", [(64, 32), (40, 25)])
def test_two_rank_gloo_shard_and_gather(ob, cornell, w, h):
    """world_size-2 gloo: image sharding + all_gather reassembles the single-device image bit for bit;
    frame sharding + reduce(sum) equals the sum of the two single frames."""
    import socket
    import torch.multiprocessing as mp

    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, w, h, 64, q)) for r in range(2)]
    for p in procs:
        p.start()
    img_bytes, acc_bytes = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    tris, mats = cornell
    full, _, _ = ob.render(ob.default_params(w, h, n_frames=2, mode=3, accum=1, max_depth=4), tris, mats)
    assert img_bytes == full.tobytes()
    f0, _, _ = ob.render(ob.default_params(w, h, first_frame=0, n_frames=1, mode=3, accum=1, max_depth=4), tris, mats)
    f1, _, _ = ob.render(ob.default_params(w, h, first_frame=1, n_frames=1, mode=3, accum=1, max_depth=4), tris, mats)
    assert acc_bytes == (f0 + f1).tobytes()


def test_bench_reference_arm_runs_without_gpu():
    """bench.py --impl reference times the oracle port on the host cores and prints the contract's JSON line."""
    import json
    import subprocess
    import sys
    from conftest import ROOT
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--workload", "c2"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "Mrays/s" and d["value"] > 0 and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] == len(os.sched_getaffinity(0))
    assert d["e2e"] == {"value": d["value"], "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"].startswith("c2")
    import bench
    assert d["config"] == bench.config_of("c2", 1)  # the same `config` as this repo's arm prints for that workload


def test_bench_refuses_without_gpu():
    import subprocess
    import sys
    import torch
    from conftest import ROOT
    if torch.cuda.is_available():
        pytest.skip("needs a CPU-only host")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"], capture_output=True, text=True, timeout=300)
    assert r.returncode != 0 and "no CUDA device" in (r.stderr + r.stdout)


def test_unmodified_reference_test_over_shim_needs_a_device(pt, tmp_path):
    """oracle/_ref/adlTest64_ptb200 (the reference's own test sources compiled against the ADL-shaped shim) links
    libptb200.so and has no CPU path: without a device its fixture cannot allocate one and every case fails."""
    import subprocess
    exe = os.path.join(ROOT, "oracle", "_ref", "adlTest64_ptb200")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/adlTest64_ptb200 not built (make -C oracle ref needs the reference tree)")
    n = C.c_int(-1)
    if pt.lib().ptb_device_count(C.byref(n)) == 0 and n.value > 0:
        pytest.skip("a CUDA device is present")
    ldd = subprocess.run(["ldd", exe], capture_output=True, text=True).stdout
    assert "libptb200.so" in ldd and "libOpenCL" not in ldd
    env = dict(os.environ, PTB_REF_WORKDIR=str(tmp_path / "ref"))
    r = subprocess.run([exe, "--gtest_filter=DeviceTest.initialize:DeviceTest.deviceInfo"], capture_output=True, text=True, timeout=60, env=env)
    assert r.returncode != 0 and "FAILED" in r.stdout


def test_bench_reference_arm_under_torchrun():
    """Launched like the driver does for N>1: rank 0 alone runs and prints the line, the other ranks exit 0 silently."""
    import json
    import subprocess
    import sys
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29641", os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                        "--warmup", "0"], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 2 and d["value"] > 0
    # torchrun exports OMP_NUM_THREADS=1 to its workers: the arm must still use every host core it may run on
    assert d["cpu_baseline"]["cores"] == len(os.sched_getaffinity(0))
    assert len(os.sched_getaffinity(0)) == 1 or d["cpu_baseline"]["cores"] > 1
    import bench
    assert d["config"] == bench.config_of("c5", 2) and d["config"]["workload"].startswith("c5")  # default workload, same config as our arm


def test_bench_dump_outputs_samples_large_images(tmp_path):
    """bench.py --dump-outputs: an image larger than DUMP_PIXELS is written as the rows of a fixed sample of distinct pixels in
    ascending order, identical from run to run and far below 64 MB; a smaller one is written whole."""
    import bench
    n = bench.DUMP_PIXELS + 1_000_000
    img = np.arange(n * 4, dtype=np.float32).reshape(n, 4)  # row k holds 4k .. 4k+3, exact in float32
    bench.dump_outputs(str(tmp_path / "a"), img)
    bench.dump_outputs(str(tmp_path / "b"), img)
    a, b = np.load(tmp_path / "a" / "image.npy"), np.load(tmp_path / "b" / "image.npy")
    assert a.dtype == np.float32 and a.shape == (bench.DUMP_PIXELS, 4) and a.nbytes <= 64 << 20
    assert a.tobytes() == b.tobytes()
    rows = a[:, 0].astype(np.int64) // 4
    assert (np.diff(rows) > 0).all() and rows[0] >= 0 and rows[-1] < n
    np.testing.assert_array_equal(a, img[rows])
    bench.dump_outputs(str(tmp_path / "c"), img[:1000])
    assert np.load(tmp_path / "c" / "image.npy").tobytes() == img[:1000].tobytes()
