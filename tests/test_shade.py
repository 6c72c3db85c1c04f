"""ptb_scene_shade: render-mode samples (PRIMARY, AO, DIRECT, PATH) along caller-owned device rays.

CPU: the record layout, argument checks that need no device, the resource usage of the C5 buffer-source path kernel, and the
reference for samples on arbitrary rays (tests/oracle_shade.c: the oracle's own per-sample integrators called with ray i and
seed i), pinned to ora_render on the oracle's camera rays.
GPU: bit-exact against ptb_render on its own camera rays and seeds, against the oracle on rays no camera makes, through torch
tensors, over ragged sizes and bad arguments, and without device-memory growth.
"""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from conftest import ROOT, assert_same_tree, bits, oracle_params, oracle_tree

STAT_FIELDS = ("tri", "quad", "t_bits", "visits_primary", "visits_secondary", "count", "id_hash", "tri_tests")
CTR_FIELDS = ("rays_closest", "rays_any", "nodes", "tri_tests", "samples")
MODES = (0, 1, 2, 3)  # PRIMARY, AO, DIRECT, PATH


# ---- no device needed --------------------------------------------------------------------------------

def test_sample_ray_dtype_matches_the_header(pt, tmp_path):
    src = tmp_path / "layout.c"
    src.write_text(
        '#include <stddef.h>\n#include <stdio.h>\n#include "SharedHeader.h"\n'
        "int main(void) {\n"
        '  printf("%zu %zu %zu %zu %zu\\n", sizeof(ptb_sample_ray), offsetof(ptb_sample_ray, o), offsetof(ptb_sample_ray, seed), '
        "offsetof(ptb_sample_ray, d), offsetof(ptb_sample_ray, reserved));\n"
        "  return 0;\n}\n")
    exe = tmp_path / "layout"
    subprocess.check_call(["cc", "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = list(map(int, subprocess.check_output([str(exe)], text=True).split()))
    R = pt.SAMPLE_RAY_DTYPE
    assert got == [R.itemsize] + [R.fields[f][1] for f in ("o", "seed", "d", "reserved")] == [32, 0, 12, 16, 28]
    assert R.fields["seed"][0] == np.dtype("<u4")


def test_shade_null_handles_are_refused_without_a_device(pt):
    L = pt.lib()
    assert L.ptb_scene_shade(None, None, None, None, 16, None, None, None) == -1  # PTB_E_INVALID
    assert b"ptb_scene_shade" in L.ptb_last_error() and b"null" in L.ptb_last_error()


@pytest.fixture(scope="module")
def ora_shade(ob, tmp_path_factory):
    """ora_shade(prm, tris, mats, o, d, seeds, bvh) -> (float4 per ray, stats per ray, counters dict)"""
    out = tmp_path_factory.mktemp("oracle_shade") / "liboracle_shade.so"
    cc = shutil.which("gcc", path="/usr/bin") or "gcc"  # the compiler and flags of oracle/Makefile
    subprocess.check_call([cc, "-O2", "-std=c11", "-fPIC", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-fno-math-errno",
                           "-mfma", "-shared", "-I", os.path.join(ROOT, "oracle"), "-o", str(out),
                           os.path.join(ROOT, "tests", "oracle_shade.c"), os.path.join(ROOT, "oracle", "oracle_bvh.c"), "-lm"])
    lib = C.CDLL(str(out))
    lib.ora_shade.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int] + [C.c_void_p] * 6

    def run(prm, tris, mats, o, d, seeds, bvh=None):
        n = len(o)
        prm.use_bvh = 1 if bvh is not None else 0
        tris, mats = np.ascontiguousarray(tris), np.ascontiguousarray(mats)
        o, d = np.ascontiguousarray(o, np.float32), np.ascontiguousarray(d, np.float32)
        seeds = np.ascontiguousarray(seeds, np.uint32)
        rad = np.zeros((n, 4), np.float32)
        st = np.zeros(n, ob.STATS_DTYPE)
        ctr = ob.Counters()
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        rc = lib.ora_shade(C.byref(prm), p(tris), len(tris), p(mats), C.cast(C.byref(bvh), C.c_void_p) if bvh is not None else None,
                           n, p(o), p(d), p(seeds), p(rad), p(st), C.byref(ctr))
        assert rc == 0
        return rad, st, ctr.as_dict()

    return run


def _oracle_camera(ob, w, h, frame, gids):
    """the oracle's camera rays and post-camera seeds (GenerateColors.cl:305-310)"""
    o, d, s = np.empty((len(gids), 3), np.float32), np.empty((len(gids), 3), np.float32), np.empty(len(gids), np.uint32)
    h32 = ob.lib().ora_hash_uint32(frame)
    for i, g in enumerate(gids):
        o[i], d[i], s[i] = ob.generate_ray(int(g) % w, int(g) // w, w, h, (int(g) + h32) & 0xFFFFFFFF)
    return o, d, s


@pytest.mark.parametrize("form", ["brute", 1, 4, 2])
def test_oracle_shade_on_camera_rays_is_ora_render(ob, cornell, ora_shade, form):
    """the reference pins itself: on the camera rays and seeds of frame 3 it reproduces a one-frame ACCUM_LINEAR ora_render bit
    for bit (image, statistics, counters) in every mode, on the FLAT, 4-wide and binary trees and brute force"""
    tris, mats = cornell
    bvh = None
    if form != "brute":
        bvh, _keep, _b = oracle_tree(ob, tris, width=form)
    w, h, frame = 64, 48, 3
    gids = np.arange(w * h)
    o, d, s = _oracle_camera(ob, w, h, frame, gids)
    for mode in MODES:
        prm = oracle_params(ob, tris, w, h, first_frame=frame, n_frames=1, mode=mode, accum=ob.ACCUM_LINEAR, max_depth=8,
                            ao_samples=4, use_bvh=1 if bvh is not None else 0)
        fb, st, ctr = ob.render(prm, tris, mats, bvh=bvh, want_stats=True)
        rad, st2, ctr2 = ora_shade(prm, tris, mats, o, d, s, bvh)
        np.testing.assert_array_equal(bits(rad), bits(fb), err_msg=f"mode {mode}")
        assert st2.tobytes() == st.tobytes(), f"mode {mode}"
        assert ctr2 == ctr, f"mode {mode}"
        assert ctr["rays_closest"] >= w * h


def _cuobjdump():
    found = shutil.which("cuobjdump")
    if found:
        return found
    cuda = os.environ.get("CUDA_HOME") or os.environ.get("CUDA_PATH") or "/usr/local/cuda"
    return os.path.join(cuda, "bin", "cuobjdump")


def test_buffer_source_c5_path_kernel_has_no_spills(pt):
    """the C5 path kernel on a caller's rays keeps the camera form's budget: no local memory, the traversal stack alone as its
    stack frame, and registers that allow the 11 CTAs of 128 threads per SM of its launch bound"""
    out = subprocess.run([_cuobjdump(), "--dump-resource-usage", pt.LIB_PATH], check=True, capture_output=True, text=True).stdout
    usage = dict(re.findall(r"Function (_ZN3ptd15k_path_sm2_raysILb0ELi11ELi6E\S*):\s*\n\s*(REG:.*)", out))
    assert len(usage) == 1, "the buffer-source C5 path kernel is missing from libptb200.so"
    u = {k: int(v) for k, v in re.findall(r"(\w+):(\d+)", next(iter(usage.values())))}
    with open(os.path.join(ROOT, "oclpathtracer_b200", "csrc", "pt_device.cuh")) as f:
        stack = (int(re.search(r"#define PTD_LSTACK_ENTRIES (\d+)", f.read()).group(1)) + 1) * 8
    assert u["LOCAL"] == 0 and u["STACK"] == stack == 1032
    per_warp = -(-u["REG"] * 32 // 256) * 256
    assert 65536 // (per_warp * 4) >= 11, u["REG"]


# ---- on the B200 -------------------------------------------------------------------------------------

def _pack(o, d, seeds):
    r = np.zeros(len(o), np.dtype([("o", "<f4", 3), ("seed", "<u4"), ("d", "<f4", 3), ("reserved", "<i4")]))
    r["o"], r["seed"], r["d"] = o, seeds, d
    return r


def _shade(dev, pt, scene, prm, o, d, seeds, stats=True):
    """Buffer path -> (radiance float32 (n, 4), stats STATS_DTYPE or None, counters)"""
    n = len(o)
    rb, ob_ = dev.buffer(max(1, n) * 32), dev.buffer(max(1, n) * 16)
    sb = dev.buffer(max(1, n) * 32) if stats else None
    if n:
        rb.write(_pack(o, d, seeds))
        _, ctr = dev.shade(scene, prm, rb, ob_, stats=sb, want_counters=True)
    else:  # a Buffer's size gives Device.shade its ray count: call the C entry point with n = 0
        c = pt.Counters()
        assert pt.lib().ptb_scene_shade(dev.handle, scene._h, C.byref(prm), rb._h, 0, ob_._h, sb._h if sb is not None else None,
                                        C.byref(c)) == 0
        ctr = c.as_dict()
    rad = ob_.read(np.float32, count=4 * n).reshape(-1, 4)
    st = sb.read(pt.STATS_DTYPE, count=n) if stats else None
    for b in (rb, ob_, sb):
        if b is not None:
            b.close()
    return rad, st, ctr


def _render(dev, pt, scene, w, h, frame, mode, max_depth=8, ao_samples=16, tuning=()):
    prm = pt.default_params(width=w, height=h, first_frame=frame, n_frames=1, mode=mode, accum=pt.ACCUM_LINEAR,
                            collect_stats=1, max_depth=max_depth, ao_samples=ao_samples)
    fb, sb = dev.buffer(w * h * 16), dev.buffer(w * h * 32)
    ctr = dev.render(scene, prm, fb, sb, want_counters=True)
    rad, st = fb.read(np.float32).reshape(-1, 4), sb.read(pt.STATS_DTYPE)
    fb.close(); sb.close()
    return prm, rad, st, ctr


def _assert_same(rad, st, ctr, rad2, st2, ctr2, msg):
    np.testing.assert_array_equal(bits(rad), bits(rad2), err_msg=f"{msg} radiance")
    if st is not None and st2 is not None:
        for f in STAT_FIELDS:
            np.testing.assert_array_equal(st[f], st2[f], err_msg=f"{msg} {f}")
    for f in CTR_FIELDS:
        if ctr is not None and ctr2 is not None and (f not in ("nodes", "tri_tests") or (st is not None and st2 is not None)):
            assert ctr[f] == ctr2[f], (msg, f, ctr[f], ctr2[f])


@pytest.fixture(scope="module")
def tess(pt, cornell):
    tris, _ = cornell
    return pt.tessellate(tris, 12)  # 5184 triangles: binary tree traversed from L2/HBM


def _equals_render(dev, pt, sc, w, h, frame, mode, max_depth=8, stats=True, msg=""):
    prm, rad, st, ctr = _render(dev, pt, sc, w, h, frame, mode, max_depth=max_depth)
    o, d, s = dev.test_camera(w, h, frame, np.arange(w * h, dtype=np.int32))
    rad2, st2, ctr2 = _shade(dev, pt, sc, prm, o, d, s, stats=stats)
    _assert_same(rad, st if stats else None, ctr, rad2, st2, ctr2, f"{msg} mode {mode} depth {max_depth}")
    return ctr2


@pytest.mark.gpu
def test_shade_equals_render_on_the_cornell_box(dev, pt, cornell, tess):
    tris, mats = cornell
    sc = dev.scene(tris, mats)
    assert sc.info()["width"] == 1
    for mode in MODES:
        _equals_render(dev, pt, sc, 96, 64, 5, mode, msg="flat")
    for depth in (1, 16):
        _equals_render(dev, pt, sc, 96, 64, 2, pt.MODE_PATH, max_depth=depth, msg="flat")
    sc.close()
    sc4 = dev.scene(tris, mats, pt.bvh_params(force_width=4))
    assert sc4.info()["width"] == 4
    for mode in (pt.MODE_AO, pt.MODE_PATH):
        _equals_render(dev, pt, sc4, 96, 64, 1, mode, msg="wide4")
    sc4.close()
    for gpu in (False, True):
        st = dev.scene(tess, mats, gpu_build=gpu)
        assert st.info()["width"] == 2
        for mode in (MODES if not gpu else (pt.MODE_PATH,)):
            _equals_render(dev, pt, st, 96, 64, 4, mode, msg=f"tess gpu={gpu}")
        st.close()


@pytest.mark.gpu
def test_shade_equals_render_on_c5(dev, pt, cornell):
    """2M triangles, 1024^2 camera rays, PATH depth 8: k_path_sm2_rays with and without statistics, and the k_mega_path_regen
    fallback when the traversal stack lives in shared memory (tuning knob 2 = 2)"""
    tris, mats = cornell
    sc = dev.scene(pt.tessellate(tris, 236), mats)
    for stats in (False, True):
        ctr = _equals_render(dev, pt, sc, 1024, 1024, 7, pt.MODE_PATH, stats=stats, msg=f"c5 stats={stats}")
        assert ctr["samples"] == 1024 * 1024
    sc.close()
    dev.set_tuning(2, 2)
    try:
        sc = dev.scene(pt.tessellate(tris, 236), mats)
        _equals_render(dev, pt, sc, 1024, 1024, 7, pt.MODE_PATH, msg="c5 shared-memory stack")
        sc.close()
    finally:
        dev.set_tuning(2, 0)


def _odd_rays(n, seed):
    """rays no camera makes: origins inside the box, origins far outside aimed in, axis-parallel directions, random seeds"""
    rng = np.random.default_rng(seed)
    o = rng.uniform([-0.9, 0.1, -0.9], [0.9, 5.4, 3.9], (n, 3)).astype(np.float32)
    d = rng.normal(size=(n, 3))
    d = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)
    k = n // 8
    d[:k] = np.float32([0, 0, -1])
    d[k:2 * k] = np.float32([0, -1, 0])
    d[2 * k:3 * k] = np.float32([1, 0, 0])
    far = slice(3 * k, 5 * k)
    o[far] = rng.uniform(-1, 1, (2 * k, 3)) * np.float32(300.0)
    v = rng.uniform([-1, 0.5, -1], [1, 5, 1], (2 * k, 3)) - o[far]
    d[far] = (v / np.linalg.norm(v, axis=1, keepdims=True)).astype(np.float32)
    seeds = rng.integers(0, 1 << 32, n, dtype=np.uint64).astype(np.uint32)
    return o, d, seeds


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["flat", "wide4", "sah", "lbvh"])
def test_shade_equals_the_oracle_on_arbitrary_rays(dev, pt, ob, cornell, tess, ora_shade, case):
    tris, mats = cornell
    for mode in MODES:
        if case == "flat":
            sc, stris = dev.scene(tris, mats), tris
            width = sc.mode_width(mode)
            bvh, _keep, ot = oracle_tree(ob, tris, width=width)
        elif case == "wide4":
            sc, stris = dev.scene(tris, mats, pt.bvh_params(force_width=4)), tris
            bvh, _keep, ot = oracle_tree(ob, tris, width=4)
        elif case == "sah":
            sc, stris = dev.scene(tess, mats), tess
            bvh, _keep, ot = oracle_tree(ob, tess, width=2)
        else:
            sc, stris = dev.scene(tess, mats, gpu_build=True), tess
            bvh, _keep = ob.make_bvh(*sc.bvh())
            ot = None
        if ot is not None:
            if sc.mode_width(mode) == sc.info()["width"]:
                assert_same_tree(*sc.bvh(), ot)
            assert ot["width"] == sc.mode_width(mode)
        o, d, s = _odd_rays(20_000, 80 + mode)
        prm = pt.default_params(mode=mode, max_depth=8, ao_samples=8)
        oprm = oracle_params(ob, stris, 1, 1, mode=mode, max_depth=8, ao_samples=8)
        rad, st, ctr = _shade(dev, pt, sc, prm, o, d, s)
        want_rad, want_st, want_ctr = ora_shade(oprm, stris, mats, o, d, s, bvh)
        np.testing.assert_array_equal(bits(rad), bits(want_rad), err_msg=f"{case} mode {mode}")
        assert st.tobytes() == want_st.tobytes(), f"{case} mode {mode}"
        for f in CTR_FIELDS:
            assert ctr[f] == want_ctr[f], (case, mode, f)
        assert (st["tri"] == -1).any() and (st["tri"] >= 0).any()
        sc.close()


@pytest.mark.gpu
def test_shade_on_torch_tensors(pt, cornell, tess):
    torch = pytest.importorskip("torch")
    tris, mats = cornell
    dev = pt.Device(0, stream=torch.cuda.current_stream().cuda_stream)
    try:
        sc = dev.scene(tess, mats)
        o, d, s = _odd_rays(30_000, 90)
        prm = pt.default_params(mode=pt.MODE_PATH, max_depth=8)
        want_rad, want_st, _ = _shade(dev, pt, sc, prm, o, d, s)
        rays = torch.from_numpy(_pack(o, d, s).view(np.int32).reshape(-1, 8)).cuda()
        rad = torch.full((len(o), 4), -7.0, dtype=torch.float32, device="cuda")
        st = torch.zeros((len(o), 8), dtype=torch.int32, device="cuda")
        out = dev.shade(sc, prm, rays, rad, stats=st)
        assert out is rad
        np.testing.assert_array_equal(rad.cpu().numpy().view(np.uint32), bits(want_rad))
        assert st.cpu().numpy().tobytes() == want_st.tobytes()
        # float32 rays with the seed's bits, and radiance allocated by the binding
        r2 = dev.shade(sc, prm, rays.view(torch.float32))
        assert torch.equal(r2.view(torch.int32), rad.view(torch.int32))
        # bad shapes and dtypes
        with pytest.raises(pt.PtbError, match="shape"):
            dev.shade(sc, prm, rays[:, :4].contiguous())
        with pytest.raises(pt.PtbError, match="4-byte"):
            dev.shade(sc, prm, rays.to(torch.int64))
        with pytest.raises(pt.PtbError, match="radiance"):
            dev.shade(sc, prm, rays, torch.empty((len(o), 3), dtype=torch.float32, device="cuda"))
        with pytest.raises(pt.PtbError, match="stats"):
            dev.shade(sc, prm, rays, rad, stats=torch.empty((len(o), 8), dtype=torch.float32, device="cuda"))
        # a misaligned view of the rays is refused
        flat = torch.zeros(8 * 64 + 8, dtype=torch.int32, device="cuda")
        with pytest.raises(pt.PtbError, match="aligned"):
            dev.shade(sc, prm, flat[1:1 + 8 * 64].view(64, 8))
        sc.close()
    finally:
        dev.close()
    own = pt.Device(0)
    try:
        sc = own.scene(tris, mats)
        with pytest.raises(pt.PtbError, match="current_stream"):
            own.shade(sc, pt.default_params(), torch.zeros((4, 8), dtype=torch.int32, device="cuda"))
        sc.close()
    finally:
        own.close()


@pytest.mark.gpu
def test_shade_ragged_sizes_and_refusals(dev, pt, ob, cornell, ora_shade):
    tris, mats = cornell
    flat = dev.scene(tris, mats)
    c5 = dev.scene(pt.tessellate(tris, 236), mats)
    prm = pt.default_params(mode=pt.MODE_PATH, max_depth=8)
    bvh, _keep, _b = oracle_tree(ob, tris, width=1)
    oprm = oracle_params(ob, tris, 1, 1, mode=ob.MODE_PATH, max_depth=8)
    for n in (0, 1, 31, 129, (1 << 20) + 7):
        o, d, s = _odd_rays(max(n, 8), 100 + (n & 1023))
        o, d, s = o[:n], d[:n], s[:n]
        for sc in (flat, c5):
            rad, st, ctr = _shade(dev, pt, sc, prm, o, d, s)
            assert ctr["samples"] == n and ctr["rays_closest"] == int(st["count"].sum())
            assert ctr["nodes"] == int(st["visits_primary"].sum() + st["visits_secondary"].sum())
            assert ctr["tri_tests"] == int(st["tri_tests"].sum())
            if n and sc is flat and n < 1000:
                want, want_st, _ = ora_shade(oprm, tris, mats, o, d, s, bvh)
                np.testing.assert_array_equal(bits(rad), bits(want), err_msg=f"n={n}")
                assert st.tobytes() == want_st.tobytes()
    # every refusal, by return code and message
    L = pt.lib()
    rb, rad, st, tiny = dev.buffer(32 * 100), dev.buffer(16 * 100), dev.buffer(32 * 100), dev.buffer(16 * 50)
    big = dev.buffer(32 * 101 + 32)
    mis_r = dev.wrap(pt.lib().ptb_buffer_device_ptr(big._h) + 16, 32 * 100)
    mis_o = dev.wrap(pt.lib().ptb_buffer_device_ptr(big._h) + 8, 16 * 100)

    def call(p=prm, r=rb, n=100, o=rad, s=None, scene=flat, device=dev):
        h = lambda x: x._h if x is not None else None
        return L.ptb_scene_shade(device.handle if device is not None else None, h(scene), C.byref(p) if p is not None else None,
                                 h(r), n, h(o), h(s), None)

    def P(**kw):
        q = pt.default_params(mode=pt.MODE_PATH, max_depth=8)
        for k, v in kw.items():
            setattr(q, k, v)
        return q

    cases = [
        (dict(device=None), b"null"), (dict(scene=None), b"null"), (dict(p=None), b"null"), (dict(r=None), b"null"),
        (dict(o=None), b"null"), (dict(n=-1), b"< 0"), (dict(p=P(mode=4)), b"bad mode"), (dict(p=P(mode=-1)), b"bad mode"),
        (dict(p=P(max_depth=0)), b"bad max_depth"), (dict(p=P(max_depth=4097)), b"bad max_depth"),
        (dict(p=P(mode=pt.MODE_AO, ao_samples=0)), b"bad ao_samples"), (dict(p=P(mode=pt.MODE_AO, ao_samples=4097)), b"bad ao_samples"),
        (dict(p=P(mode=pt.MODE_DIRECT, light_quad=99)), b"light_quad"), (dict(p=P(mode=pt.MODE_DIRECT, light_quad=-1)), b"light_quad"),
        (dict(p=P(accel=pt.ACCEL_BRUTE)), b"accel"), (dict(p=P(integrator=pt.INTEGRATOR_WAVEFRONT)), b"integrator"),
        (dict(n=101), b"rays buffer too small"), (dict(o=tiny), b"radiance buffer too small"), (dict(s=tiny), b"stats buffer too small"),
        (dict(r=mis_r), b"32-byte aligned"), (dict(o=mis_o), b"16-byte aligned"), (dict(s=mis_o, n=50), b"16-byte aligned"),
    ]
    for kw, msg in cases:
        assert call(**kw) == -1, kw
        err = L.ptb_last_error()
        assert b"ptb_scene_shade" in err and msg in err, (kw, err)
    assert call(n=0) == 0 and call() == 0 and call(s=st) == 0
    other = pt.Device(0)
    osc = other.scene(tris, mats)
    ob_ = other.buffer(32 * 100)
    assert call(scene=osc) == -1 and b"scene belongs to another device" in L.ptb_last_error()
    assert call(r=ob_) == -1 and b"buffer belongs to another device" in L.ptb_last_error()
    ob_.close(); osc.close(); other.close()
    dev.sync()
    for b in (mis_r, mis_o, big, rb, rad, st, tiny):
        b.close()
    # counters in cumulative mode add up over a render call and shade calls
    o, d, s = _odd_rays(5000, 120)
    prm_ao = pt.default_params(width=32, height=32, n_frames=1, mode=pt.MODE_AO, accum=pt.ACCUM_LINEAR)
    frame = dev.buffer(32 * 32 * 16)
    want_r = dev.render(flat, prm_ao, frame, None, want_counters=True)
    _, _, want_s = _shade(dev, pt, flat, prm_ao, o, d, s)
    dev.counters(cumulative=1, read=False)
    try:
        dev.render(flat, prm_ao, frame, None)
        _shade(dev, pt, flat, prm_ao, o, d, s)
        tot = dev.counters(read=True)
    finally:
        dev.counters(cumulative=0, read=False)
    frame.close()
    for f in ("rays_closest", "rays_any", "samples"):
        assert tot[f] == want_r[f] + want_s[f], f
    flat.close(); c5.close()


@pytest.mark.gpu
def test_shade_leaks_no_device_memory(pt, cornell, tess):
    tris, mats = cornell
    probe = pt.Device(0)
    free0 = None
    o, d, s = _odd_rays(200_000, 130)
    for it in range(5):
        dv = pt.Device(0)
        for sc in (dv.scene(tris, mats), dv.scene(tess, mats)):
            for mode in MODES:
                _shade(dv, pt, sc, pt.default_params(mode=mode, max_depth=8), o, d, s, stats=mode % 2 == 0)
            sc.close()
        dv.close()
        free, _ = probe.memory()
        if it == 1:
            free0 = free
        elif it > 1:
            assert free >= free0 - (8 << 20), (it, free0, free)
    probe.close()
