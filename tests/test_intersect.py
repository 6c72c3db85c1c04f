"""ptb_scene_intersect: closest- and any-hit queries on caller-owned device ray buffers.

CPU: the record layouts, argument checks that need no device, and the reference for closest hits with a per-ray tmax
(tests/oracle_tmax.c: the oracle's own traversal called with tmax[i] where ora_trace passes 1e20).
GPU: bit-exact against the oracle walking its own tree of each form (tri, t, u, v, node visits, triangle tests), against
ptb_trace on the 2M-triangle scene, against the PRIMARY render statistics, through torch tensors, and over ragged sizes.
"""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

from conftest import ROOT, assert_same_tree, bits, oracle_tree

FIELDS = ("tri", "t", "u", "v", "visits", "tests")


# ---- no device needed --------------------------------------------------------------------------------

def test_ray_and_hit_dtypes_match_the_header(pt, tmp_path):
    src = tmp_path / "layout.c"
    src.write_text(
        '#include <stddef.h>\n#include <stdio.h>\n#include "SharedHeader.h"\n'
        "int main(void) {\n"
        '  printf("%zu %zu %zu %zu %zu\\n", sizeof(ptb_ray), offsetof(ptb_ray, o), offsetof(ptb_ray, tmax), offsetof(ptb_ray, d), offsetof(ptb_ray, reserved));\n'
        '  printf("%zu %zu %zu %zu %zu\\n", sizeof(ptb_hit), offsetof(ptb_hit, t), offsetof(ptb_hit, u), offsetof(ptb_hit, v), offsetof(ptb_hit, tri));\n'
        '  printf("%d %d\\n", PTB_QUERY_CLOSEST, PTB_QUERY_ANY);\n'
        "  return 0;\n}\n")
    exe = tmp_path / "layout"
    subprocess.check_call(["cc", "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    ray, hit, q = [list(map(int, l.split())) for l in subprocess.check_output([str(exe)], text=True).splitlines()]
    R, H = pt.RAY_DTYPE, pt.HIT_DTYPE
    assert ray == [R.itemsize] + [R.fields[f][1] for f in ("o", "tmax", "d", "reserved")] == [32, 0, 12, 16, 28]
    assert hit == [H.itemsize] + [H.fields[f][1] for f in ("t", "u", "v", "tri")] == [16, 0, 4, 8, 12]
    assert q == [pt.QUERY_CLOSEST, pt.QUERY_ANY]


def test_intersect_null_handles_are_refused_without_a_device(pt):
    L = pt.lib()
    assert L.ptb_scene_intersect(None, None, 0, None, 16, None, None, None) == -1  # PTB_E_INVALID
    assert b"ptb_scene_intersect" in L.ptb_last_error() and b"null" in L.ptb_last_error()


def _rays(n, seed):
    """the parity tests' generator (axis-parallel and NaN directions) plus origins far outside the scene aiming at it"""
    rng = np.random.default_rng(seed)
    o = rng.uniform([-2.7, 0.05, -5.5], [2.7, 5.4, 3.9], (n, 3)).astype(np.float32)
    d = rng.normal(size=(n, 3))
    d = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)
    d[:64] = np.float32([0, 0, -1])
    d[64:128] = np.float32([0, -1, 0])
    d[128:192] = np.float32([-1, 0, 0])
    d[192:200] = np.float32([np.nan, 0, 1])
    far = slice(200, 400)
    o[far] = rng.uniform(-1, 1, (200, 3)) * np.float32(500.0)
    tgt = rng.uniform([-1, 0.5, -1], [1, 5, 1], (200, 3))
    v = tgt - o[far]
    d[far] = (v / np.linalg.norm(v, axis=1, keepdims=True)).astype(np.float32)
    return o, d


def _tmax_mix(rng, hit_t, n):
    """per-ray tmax from {1e20, random, exactly the closest hit's t (strict <: a miss), 0, negative, NaN}"""
    kind = rng.integers(0, 6, n)
    tm = np.full(n, 1e20, np.float32)
    tm[kind == 1] = rng.uniform(0.0, 6.0, (kind == 1).sum()).astype(np.float32)
    exact = (kind == 2) & (hit_t > 0)
    tm[exact] = hit_t[exact]
    tm[kind == 3] = 0.0
    tm[kind == 4] = -rng.uniform(0.0, 5.0, (kind == 4).sum()).astype(np.float32)
    tm[kind == 5] = np.nan
    return tm, exact


@pytest.fixture(scope="module")
def closest_tmax(ob, tmp_path_factory):
    """closest_tmax(tris, o, d, tmax, bvh) -> dict like ob.trace's: the oracle's closest-hit query with a per-ray tmax"""
    out = tmp_path_factory.mktemp("oracle_tmax") / "liboracle_tmax.so"
    cc = shutil.which("gcc", path="/usr/bin") or "gcc"  # the compiler and flags of oracle/Makefile
    subprocess.check_call([cc, "-O2", "-std=c11", "-fPIC", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-fno-math-errno",
                           "-mfma", "-shared", "-I", os.path.join(ROOT, "oracle"), "-o", str(out),
                           os.path.join(ROOT, "tests", "oracle_tmax.c"), os.path.join(ROOT, "oracle", "oracle_bvh.c"), "-lm"])
    lib = C.CDLL(str(out))
    lib.ora_trace_closest_tmax.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int] + [C.c_void_p] * 9

    def run(tris, o, d, tmax, bvh=None):
        n = len(o)
        tris = np.ascontiguousarray(tris)
        o, d = np.ascontiguousarray(o, np.float32), np.ascontiguousarray(d, np.float32)
        tmax = np.ascontiguousarray(np.broadcast_to(np.asarray(tmax, np.float32), (n,)))
        r = {"tri": np.empty(n, np.int32), "t": np.empty(n, np.float32), "u": np.empty(n, np.float32), "v": np.empty(n, np.float32),
             "visits": np.empty(n, np.uint32), "tests": np.empty(n, np.uint32)}
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        lib.ora_trace_closest_tmax(p(tris), len(tris), C.cast(C.byref(bvh), C.c_void_p) if bvh is not None else None, n, p(o), p(d),
                                   p(tmax), *[p(r[k]) for k in FIELDS])
        return r

    return run


@pytest.mark.parametrize("form", ["brute", 1, 4, 2])
def test_oracle_closest_hit_honours_tmax(ob, cornell, closest_tmax, form):
    """the reference closest hit with a per-ray tmax == ora_trace's closest hit at 1e20 where t < tmax, a miss elsewhere;
    at tmax = 1e20 it is ora_trace itself, node visits and triangle tests included"""
    tris, _ = cornell
    bvh = None
    if form != "brute":
        bvh, _keep, _b = oracle_tree(ob, tris, width=form)
    o, d = _rays(20_000, 3)
    ref = ob.trace(tris, o, d, np.float32(1e20), bvh=bvh)
    for f in FIELDS:
        np.testing.assert_array_equal(bits(closest_tmax(tris, o, d, np.float32(1e20), bvh)[f]), bits(ref[f]), err_msg=f)
    tm, _ = _tmax_mix(np.random.default_rng(4), ref["t"], len(o))
    got = closest_tmax(tris, o, d, tm, bvh)
    keep = (ref["tri"] >= 0) & (ref["t"] < tm)
    assert keep.any() and (~keep).any()
    for f in ("tri", "t", "u", "v"):
        np.testing.assert_array_equal(bits(got[f])[keep], bits(ref[f])[keep], err_msg=f)
    assert (got["tri"][~keep] == -1).all()
    for f in ("t", "u", "v"):
        assert (bits(got[f])[~keep] == 0).all()


# ---- on the B200 -------------------------------------------------------------------------------------

def _pack(o, d, tmax):
    r = np.zeros((len(o), 8), np.float32)
    r[:, 0:3], r[:, 3], r[:, 4:7] = o, tmax, d
    return r


def _run(dev, scene, o, d, tmax, any_hit, stats=True, want_counters=False):
    """Buffer path: -> dict like ptb_trace's (and the counters)"""
    n = len(o)
    rb, hb = dev.buffer(n * 32), dev.buffer(n * 16)
    sb = dev.buffer(n * 8) if stats else None
    if n:
        rb.write(_pack(o, d, tmax))
    res = dev.intersect(scene, rb, hb, any_hit=any_hit, stats=sb, want_counters=want_counters)
    ctr = res[1] if want_counters else None
    h = hb.read(np.uint8, count=n * 16).view(np.float32).reshape(-1, 4)
    out = {"tri": h[:, 3].view(np.int32).copy(), "t": h[:, 0].copy(), "u": h[:, 1].copy(), "v": h[:, 2].copy()}
    if stats:
        s = sb.read(np.uint32, count=2 * n).reshape(-1, 2)
        out["visits"], out["tests"] = s[:, 0].copy(), s[:, 1].copy()
    for b in (rb, hb, sb):
        if b is not None:
            b.close()
    return (out, ctr) if want_counters else out


def _assert_same(g, r, fields=FIELDS, msg=""):
    for f in fields:
        np.testing.assert_array_equal(bits(g[f]), bits(r[f]), err_msg=f"{msg} {f}")


@pytest.fixture(scope="module")
def tess(pt, cornell):
    tris, _ = cornell
    return pt.tessellate(tris, 12)  # 5184 triangles: binary tree traversed from L2/HBM


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["flat", "wide4", "sah", "lbvh"])
def test_intersect_equals_the_oracle(dev, pt, ob, cornell, tess, closest_tmax, case):
    tris, mats = cornell
    if case == "flat":
        sc, stris = dev.scene(tris, mats), tris
        bvh, _keep, ot = oracle_tree(ob, tris)
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
    assert sc.info()["width"] == {"flat": 1, "wide4": 4, "sah": 2, "lbvh": 2}[case]
    if ot is not None:
        assert_same_tree(*sc.bvh(), ot)
    o, d = _rays(60_000, 21)
    ref = ob.trace(stris, o, d, np.float32(1e20), bvh=bvh)
    tm, exact = _tmax_mix(np.random.default_rng(22), ref["t"], len(o))
    for any_hit in (False, True):
        want = ob.trace(stris, o, d, tm, bvh=bvh, any_hit=any_hit) if any_hit else closest_tmax(stris, o, d, tm, bvh)
        got = _run(dev, sc, o, d, tm, any_hit)
        _assert_same(got, want, fields=("tri", "t", "u", "v"), msg=f"{case} any={any_hit}")
        # Node visits and tests.  One exception: any-hit rays with a NaN tmax on binary trees.  There the oracle's pop keeps a
        # deferred entry only if its entry distance is <= tmax, which is false for NaN, so it ends after its first descent.  Every
        # product kernel (ptb_trace, the AO / shadow stages, this one) never culls any-hit entries (DESIGN.md section 4) and walks
        # every box the ray enters.  Both report a miss.
        cmp = ~np.isnan(tm) if (any_hit and sc.info()["width"] == 2) else np.ones(len(o), bool)
        for f in ("visits", "tests"):
            np.testing.assert_array_equal(got[f][cmp], want[f][cmp], err_msg=f"{case} any={any_hit} {f}")
        assert (got["tri"][exact] == -1).all()  # tmax = the hit's own t: strict <
        assert (got["tri"][np.isnan(tm) | (tm <= 0)] == -1).all()
    sc.close()


@pytest.mark.gpu
def test_intersect_equals_ptb_trace_on_c5(dev, pt, cornell):
    """2M triangles, 1M rays: the persistent kernel and k_trace differ by scheduling only"""
    tris, mats = cornell
    sc = dev.scene(pt.tessellate(tris, 236), mats)
    o, d = _rays(1 << 20, 31)
    tm = np.random.default_rng(32).uniform(0.0, 4.0, len(o)).astype(np.float32)
    for any_hit, tmax in ((False, np.full(len(o), 1e20, np.float32)), (True, tm)):
        got = _run(dev, sc, o, d, tmax, any_hit)
        want = dev.trace(sc, o, d, tmax, any_hit=any_hit)
        _assert_same(got, want, msg=f"any={any_hit}")
        assert (got["tri"] >= 0).mean() > (0.2 if any_hit else 0.5)
    sc.close()


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["cornell", "tess"])
def test_intersect_equals_primary_render_statistics(dev, pt, cornell, tess, which):
    """camera rays of frame 0 (512^2): closest hit == ptb_render PRIMARY stats (tri, t bits, visits_primary)"""
    tris, mats = cornell
    sc = dev.scene(tris if which == "cornell" else tess, mats)
    w = h = 512
    o, dd, _ = dev.test_camera(w, h, 0, np.arange(w * h, dtype=np.int32))
    got = _run(dev, sc, o, dd, np.full(w * h, 1e20, np.float32), False)
    prm = pt.default_params(width=w, height=h, n_frames=1, mode=pt.MODE_PRIMARY, accum=pt.ACCUM_LINEAR, collect_stats=1)
    frame, stats = dev.buffer(w * h * 16), dev.buffer(w * h * 32)
    dev.render(sc, prm, frame, stats)
    st = stats.read(pt.STATS_DTYPE)
    frame.close(); stats.close()
    assert sc.mode_width(pt.MODE_PRIMARY) == sc.info()["width"]
    np.testing.assert_array_equal(got["tri"], st["tri"])
    np.testing.assert_array_equal(bits(got["t"]), st["t_bits"])
    np.testing.assert_array_equal(got["visits"], st["visits_primary"])
    assert (got["tri"] >= 0).all()  # every camera ray of frame 0 hits the closed box
    sc.close()


@pytest.mark.gpu
def test_intersect_on_torch_tensors(pt, cornell, tess):
    torch = pytest.importorskip("torch")
    tris, mats = cornell
    stream = torch.cuda.current_stream()
    dev = pt.Device(0, stream=stream.cuda_stream)
    try:
        sc = dev.scene(tess, mats)
        o, d = _rays(50_000, 41)
        tm = np.random.default_rng(42).uniform(0.0, 6.0, len(o)).astype(np.float32)
        rays = torch.from_numpy(_pack(o, d, tm)).cuda()
        for any_hit in (False, True):
            want = _run(dev, sc, o, d, tm, any_hit)
            hits = torch.full((len(o), 4), -7.0, dtype=torch.float32, device="cuda")
            stats = torch.zeros((len(o), 2), dtype=torch.int32, device="cuda")
            ptr = hits.data_ptr()
            out = dev.intersect(sc, rays, hits, any_hit=any_hit, stats=stats)
            assert out is hits and hits.data_ptr() == ptr
            h = hits.cpu().numpy()
            got = {"tri": hits.view(torch.int32)[:, 3].cpu().numpy(), "t": h[:, 0], "u": h[:, 1], "v": h[:, 2],
                   "visits": stats[:, 0].cpu().numpy().view(np.uint32), "tests": stats[:, 1].cpu().numpy().view(np.uint32)}
            _assert_same(got, want, msg=f"any={any_hit}")
            # hits allocated by the binding
            h2 = dev.intersect(sc, rays, any_hit=any_hit)
            assert torch.equal(h2.view(torch.int32), hits.view(torch.int32))
        # a misaligned view of the rays (a slice 4 bytes into a larger tensor) is refused
        flat = torch.zeros(8 * 64 + 8, dtype=torch.float32, device="cuda")
        with pytest.raises(pt.PtbError, match="aligned"):
            dev.intersect(sc, flat[1:1 + 8 * 64].view(64, 8))
        sc.close()
    finally:
        dev.close()
    # a Device with its own stream would race with torch's: refused
    own = pt.Device(0)
    try:
        sc = own.scene(tris, mats)
        with pytest.raises(pt.PtbError, match="current_stream"):
            own.intersect(sc, torch.zeros((4, 8), dtype=torch.float32, device="cuda"))
        sc.close()
    finally:
        own.close()


@pytest.mark.gpu
def test_intersect_shapes_errors_and_counters(dev, pt, ob, cornell, tess):
    tris, mats = cornell
    sc = dev.scene(tess, mats)
    bvh, _keep, _ot = oracle_tree(ob, tess, width=2)
    for n in (0, 1, 31, 129):
        o, d = _rays(1000, 50 + n)
        o, d = (o[-n:], d[-n:]) if n else (o[:0], d[:0])
        tm = np.full(n, 1e20, np.float32)
        for any_hit in (False, True):
            got, ctr = _run(dev, sc, o, d, tm, any_hit, want_counters=True)
            if n:
                _assert_same(got, ob.trace(tess, o, d, tm, bvh=bvh, any_hit=any_hit), msg=f"n={n}")
            assert ctr["rays_any" if any_hit else "rays_closest"] == n and ctr["rays_closest" if any_hit else "rays_any"] == 0
            assert ctr["nodes"] == int(got["visits"].sum()) and ctr["tri_tests"] == int(got["tests"].sum())
    # 2^24 + 7 rays on the FLAT scene against ptb_trace
    cs = dev.scene(tris, mats)
    n = (1 << 24) + 7
    o, d = _rays(n, 60)
    got = _run(dev, cs, o, d, np.full(n, 1e20, np.float32), False)
    _assert_same(got, dev.trace(cs, o, d, np.float32(1e20)), msg="2^24+7")
    # undersized buffers and bad arguments are refused
    rb, hb, sb, tiny = dev.buffer(32 * 100), dev.buffer(16 * 100), dev.buffer(8 * 100), dev.buffer(8 * 50)
    L = pt.lib()
    for q, r, n_, h, s, msg in ((0, rb, 101, hb, None, b"rays buffer too small"), (0, rb, 100, sb, None, b"hits buffer too small"),
                                (0, rb, 100, hb, tiny, b"stats buffer too small"), (2, rb, 100, hb, None, b"unknown query"),
                                (0, rb, -1, hb, None, b"< 0")):
        rc = L.ptb_scene_intersect(dev.handle, sc._h, q, r._h, n_, h._h, s._h if s is not None else None, None)
        assert rc == -1 and msg in L.ptb_last_error(), (q, n_, msg)
    other = pt.Device(0)
    osc = other.scene(tris, mats)
    assert L.ptb_scene_intersect(dev.handle, osc._h, 0, rb._h, 100, hb._h, None, None) == -1
    assert b"another device" in L.ptb_last_error()
    osc.close(); other.close()
    # counters in cumulative mode add up over a render call and intersect calls
    o, d = _rays(5000, 61)
    tm = np.random.default_rng(62).uniform(0.0, 5.0, len(o)).astype(np.float32)
    prm = pt.default_params(width=32, height=32, n_frames=1, mode=pt.MODE_AO, accum=pt.ACCUM_LINEAR, collect_stats=1)
    frame = dev.buffer(32 * 32 * 16)
    want_r = dev.render(sc, prm, frame, None, want_counters=True)
    dev.counters(cumulative=1, read=False)
    try:
        dev.render(sc, prm, frame, None)
        g1 = _run(dev, sc, o, d, tm, False)
        g2 = _run(dev, sc, o, d, tm, True)
        tot = dev.counters(read=True)
    finally:
        dev.counters(cumulative=0, read=False)
    frame.close()
    assert tot["rays_closest"] == want_r["rays_closest"] + len(o)
    assert tot["rays_any"] == want_r["rays_any"] + len(o)
    assert tot["nodes"] == want_r["nodes"] + int(g1["visits"].sum()) + int(g2["visits"].sum())
    assert tot["tri_tests"] == want_r["tri_tests"] + int(g1["tests"].sum()) + int(g2["tests"].sum())
    for b in (rb, hb, sb, tiny):
        b.close()
    cs.close(); sc.close()


@pytest.mark.gpu
def test_intersect_leaks_no_device_memory(pt, cornell, tess):
    tris, mats = cornell
    probe = pt.Device(0)
    free0 = None
    o, d = _rays(200_000, 70)
    tm = np.full(len(o), 1e20, np.float32)
    for it in range(5):
        dv = pt.Device(0)
        for s in (dv.scene(tris, mats), dv.scene(tess, mats)):
            for _ in range(3):
                _run(dv, s, o, d, tm, False)
                _run(dv, s, o, d, tm, True, stats=False)
            s.close()
        dv.close()
        free, _ = probe.memory()
        if it == 1:
            free0 = free
        elif it > 1:
            assert free >= free0 - (8 << 20), (it, free0, free)
    probe.close()
