"""ptb_scene_create_from_device: resident scenes built from triangle and material records already on the device.

The reference for every check is ptb_scene_create_gpu on the same records after a download: the same live nodes, tri_order,
quantised nodes, grid and ptb_scene_info, and bit for bit the same renders (every mode, megakernel and wavefront, with
statistics and counters), intersect and shade results.  The light table that replaces the host triangles of device-built
scenes equals ptb_light_from_quad on the host records.  The device-side validation gives the host loop's verdicts and names
the lowest offending triangle.
"""
import ctypes as C

import numpy as np
import pytest

from conftest import bits
from test_shade import _shade
from test_traversal_scenes import _intersect, near_rays, scene as generated_scene

EMPTY = 0x7FFFFFFF


# ---- no device needed --------------------------------------------------------------------------------

def test_null_handles_are_refused_without_a_device(pt):
    L = pt.lib()
    assert L.ptb_scene_create_from_device(None, None, 36, None, 18, None, None) == -1  # PTB_E_INVALID
    assert b"ptb_scene_create_from_device" in L.ptb_last_error() and b"null" in L.ptb_last_error()


def test_binding_declares_the_symbol(pt):
    assert "ptb_scene_create_from_device" in pt.EXPORTS
    assert pt.lib().ptb_scene_create_from_device.argtypes == [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p,
                                                              C.c_void_p]


# ---- helpers -----------------------------------------------------------------------------------------

def _upload(dev, arr):
    b = dev.buffer(arr.nbytes)
    b.write(arr)
    return b


def _from_device(dev, tris, mats, bp=None):
    tb, mb = _upload(dev, tris), _upload(dev, mats)
    try:
        return dev.scene_from_device(tb, mb, bp)
    finally:
        tb.close(); mb.close()


def _live(nodes):
    """(nodes reachable from the root, the number of levels they form); the LBVH array also holds nodes that a collapsed
    leaf hides"""
    live = np.zeros(len(nodes), bool)
    front = np.array([0])
    levels = 0
    while front.size:
        live[front] = True
        levels += 1
        ch = np.concatenate([nodes["child0"][front], nodes["child1"][front]])
        front = ch[(ch >= 0) & (ch != EMPTY)]
    return live, levels


def assert_same_scene(a, b):
    ia, ib = a.info(), b.info()
    assert ia == ib and ia["width"] == 2 and ia["smem_nodes"] == 1, (ia, ib)
    na, oa = a.bvh()
    nb, ob_ = b.bvh()
    live, levels = _live(na)
    assert np.array_equal(live, _live(nb)[0])
    assert ia["depth"] >= levels  # the traversal stack holds a path: the depth bounds the tree as traversed
    assert na[live].tobytes() == nb[live].tobytes()
    assert oa.tobytes() == ob_.tobytes()
    qa, lo_a, st_a = a.bvh_quantized()
    qb, lo_b, st_b = b.bvh_quantized()
    assert qa[live].tobytes() == qb[live].tobytes()
    assert bits(np.float32(lo_a + st_a)).tobytes() == bits(np.float32(lo_b + st_b)).tobytes()


def _with_ids(tris, n_mats):
    t = tris.copy()
    t["id"] = (np.arange(len(t)) // 2) % n_mats
    return t


def _outputs(dev, pt, sc, tris, w=40, h=32):
    """every result a scene feeds: renders of each mode and integrator (radiance, stats, counters), intersect, shade"""
    out = {}
    quad = int(tris["id"][0])  # the first pair always exists: DIRECT takes its light from the scene's light table
    for mode in (pt.MODE_PRIMARY, pt.MODE_AO, pt.MODE_DIRECT, pt.MODE_PATH):
        for integ in (pt.INTEGRATOR_MEGAKERNEL, pt.INTEGRATOR_WAVEFRONT):
            prm = pt.default_params(width=w, height=h, n_frames=2, mode=mode, accum=pt.ACCUM_LINEAR, max_depth=5, ao_samples=4,
                                    collect_stats=1, integrator=integ, light_quad=quad)
            fb, sb = dev.buffer(w * h * 16), dev.buffer(w * h * 32)
            ctr = dev.render(sc, prm, fb, sb, want_counters=True)
            out[f"render {mode} {integ}"] = (fb.read(np.uint32).tobytes(), sb.read(np.uint8).tobytes(), sorted(ctr.items()))
            fb.close(); sb.close()
    o, d = near_rays(tris, 4000, 7)
    tmax = np.random.default_rng(8).uniform(0.0, 3.0, len(o)).astype(np.float32)
    for any_hit in (False, True):
        r = _intersect(dev, sc, o, d, tmax, any_hit)
        out[f"intersect {any_hit}"] = [bits(r[f]).tobytes() for f in ("tri", "t", "u", "v", "visits", "tests")]
    seeds = np.random.default_rng(9).integers(0, 2**32, len(o), dtype=np.uint64).astype(np.uint32)
    for mode in (pt.MODE_PRIMARY, pt.MODE_AO, pt.MODE_DIRECT, pt.MODE_PATH):
        prm = pt.default_params(mode=mode, max_depth=5, ao_samples=4, light_quad=quad)
        rad, st, ctr = _shade(dev, pt, sc, prm, o, d, seeds)
        out[f"shade {mode}"] = (bits(rad).tobytes(), st.tobytes(), sorted(ctr.items()))
    return out


def assert_same_outputs(dev, pt, a, b, tris):
    ga, gb = _outputs(dev, pt, a, tris), _outputs(dev, pt, b, tris)
    assert ga.keys() == gb.keys()
    for k in ga:
        assert ga[k] == gb[k], k


CASES = {
    "cornell": (None, None),
    "tess6-leaf2": (6, 2), "tess6-leaf4": (6, 4), "tess20-leaf2": (20, 2), "tess20-leaf4": (20, 4),
    "planar-2000": ("planar-2000", None), "mixed-2000": ("mixed-2000", None), "centroid-2000": ("centroid-2000", None),
    "two-2": ("two-2", None),
}


# ---- on the B200 -------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(CASES))
def test_equals_the_host_route(dev, pt, cornell, case):
    tris, mats = cornell
    what, max_leaf = CASES[case]
    if isinstance(what, int):
        tris = pt.tessellate(tris, what)
    elif isinstance(what, str):
        tris = _with_ids(generated_scene(what), len(mats))
    bp = pt.bvh_params(max_leaf=max_leaf) if max_leaf else None
    a = dev.scene(tris, mats, bp, gpu_build=True)
    b = _from_device(dev, tris, mats, bp)
    assert b.info()["n_tris"] == len(tris) and b.info()["n_nodes"] == len(tris) - 1
    assert_same_scene(a, b)
    assert_same_outputs(dev, pt, a, b, tris)
    a.close(); b.close()


@pytest.mark.gpu
def test_c5_equals_the_host_route(dev, pt, cornell):
    """the 2,005,056-triangle C5 scene: the same tree and the same PATH samples of one shard of a 4K frame"""
    tris, mats = cornell
    big = pt.tessellate(tris, 236)
    assert len(big) == 2_005_056
    a = dev.scene(big, mats, gpu_build=True)
    b = _from_device(dev, big, mats)
    assert_same_scene(a, b)
    prm = pt.default_params(width=3840, height=2160, n_frames=1, mode=pt.MODE_PATH, accum=pt.ACCUM_LINEAR, max_depth=8,
                            collect_stats=1, shard_index=7, shard_count=64, shard_block=64)
    nl = pt.local_pixels(prm)
    got = []
    for sc in (a, b):
        fb, sb = dev.buffer(nl * 16), dev.buffer(nl * 32)
        ctr = dev.render(sc, prm, fb, sb, want_counters=True)
        got.append((fb.read(np.uint32).tobytes(), sb.read(np.uint8).tobytes(), ctr))
        fb.close(); sb.close()
    assert got[0] == got[1]
    assert got[0][2]["rays_closest"] > nl
    a.close(); b.close()


def _direct(dev, pt, sc, quad, light=None):
    kw = dict(light_p1=light[0], light_ea=light[1], light_eb=light[2]) if light else {}
    prm = pt.default_params(width=32, height=32, n_frames=1, mode=pt.MODE_DIRECT, accum=pt.ACCUM_LINEAR, collect_stats=1,
                            light_quad=quad, **kw)
    fb, sb = dev.buffer(32 * 32 * 16), dev.buffer(32 * 32 * 32)
    try:
        dev.render(sc, prm, fb, sb)
        return fb.read(np.uint32).tobytes() + sb.read(np.uint8).tobytes()
    finally:
        fb.close(); sb.close()


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["cornell", "shifted"])
def test_light_table_equals_light_from_quad(dev, pt, cornell, layout):
    """DIRECT with light_ea = 0 takes the light of light_quad from the scene's table; it equals the light ptb_light_from_quad
    derives from the host records, for every quad id, on both LBVH constructors; a quad without a pair is PTB_E_NOTFOUND with
    the host's message.  "shifted" puts one extra triangle first, so ids start at odd positions, pair with their neighbours'
    triangles or (id 17, the last) have no pair, and adds two materials no triangle uses."""
    tris, mats = cornell
    if layout == "shifted":
        tris = np.concatenate([tris[:1], tris])
        mats = np.concatenate([mats, mats[:2]])
    scenes = [_from_device(dev, tris, mats), dev.scene(tris, mats, gpu_build=True)]
    missing = 0
    for quad in range(len(mats)):
        try:
            light = pt.light_from_quad(tris, quad)
        except pt.PtbError as e:
            assert "ptb error -5" in str(e)
            missing += 1
            for sc in scenes:
                with pytest.raises(pt.PtbError) as got:
                    _direct(dev, pt, sc, quad)
                assert str(got.value) == str(e)
            continue
        want = _direct(dev, pt, scenes[0], quad, light)
        for sc in scenes:
            assert _direct(dev, pt, sc, quad) == want, quad
    assert missing == (0 if layout == "cornell" else 3)
    for sc in scenes:
        sc.close()


def _message(e):
    return str(e).split(": ", 2)[2]  # "ptb error -1: <entry point>: <verdict>"


@pytest.mark.gpu
def test_validation_names_the_lowest_offending_triangle(dev, pt, cornell):
    tris, mats = cornell
    tris = pt.tessellate(tris, 2)
    n, n_mats = len(tris), len(mats)
    tb, mb = _upload(dev, tris), _upload(dev, mats)

    def verdicts(bad):
        """(device message, host message) for records `bad`, written into the device copy in place and restored after"""
        changed = np.flatnonzero((bad.view(np.uint8).reshape(n, 64) != tris.view(np.uint8).reshape(n, 64)).any(axis=1))
        for i in changed:
            tb.write(bad[i:i + 1], offset=64 * int(i))
        try:
            with pytest.raises(pt.PtbError) as d:
                dev.scene_from_device(tb, mb)
            with pytest.raises(pt.PtbError) as h:
                dev.scene(bad, mats, gpu_build=True)
        finally:
            for i in changed:
                tb.write(tris[i:i + 1], offset=64 * int(i))
        assert "ptb_scene_create_from_device" in str(d.value) and "ptb_scene_create_gpu" in str(h.value)
        return _message(d.value), _message(h.value)

    free0 = None
    cases = 0
    for i in (0, n // 2, n - 1):
        later = min(i + 1, n - 1)
        for v in (-1, n_mats):
            bad = tris.copy()
            bad["id"][i] = v
            if later != i:
                bad["p2"][later, 1] = np.nan
            got, want = verdicts(bad)
            assert got == want == f"triangle {i} has id {v} outside [0,{n_mats})"
            cases += 1
        for f in range(12):
            for v in (np.nan, np.inf, -np.inf, 3.1e38, -3.1e38):
                bad = tris.copy()
                bad[("p1", "p2", "p3")[f // 4]][i, f % 4] = v
                if later != i:
                    bad["id"][later] = n_mats
                got, want = verdicts(bad)
                assert got == want == f"triangle {i} has a non-finite vertex", (i, f, v)
                cases += 1
        if free0 is None:
            free0 = dev.memory()[0]
    assert cases == 3 * (2 + 12 * 5)
    # the same index failing both rules: the id is reported, as the host loop checks it first
    bad = tris.copy()
    bad["id"][5] = -1
    bad["p3"][5, 3] = np.inf
    assert verdicts(bad) == ("triangle 5 has id -1 outside [0,18)",) * 2
    # +-3.0e38 is a vertex value like any other, in every float and on both routes
    ok = tris.copy()
    for f in range(12):
        ok[("p1", "p2", "p3")[f // 4]][n // 2, f % 4] = 3.0e38 if f % 2 else -3.0e38
    sc = dev.scene(ok, mats, gpu_build=True)
    tb.write(ok)
    sd = dev.scene_from_device(tb, mb)
    assert_same_scene(sc, sd)
    sc.close(); sd.close(); tb.close(); mb.close()
    assert dev.memory()[0] >= free0 - (8 << 20)


@pytest.mark.gpu
def test_two_to_the_28_triangles_are_refused_before_any_read(dev, pt, cornell):
    tris, mats = cornell
    L = pt.lib()
    h = C.c_void_p()
    t = np.ascontiguousarray(tris)
    m = np.ascontiguousarray(mats)
    assert L.ptb_scene_create_gpu(dev.handle, t.ctypes.data_as(C.c_void_p), 1 << 28, m.ctypes.data_as(C.c_void_p), len(m), None,
                                  C.byref(h)) == -1
    assert b"2^28" in L.ptb_last_error() and not h.value
    tb, mb = _upload(dev, tris), _upload(dev, mats)
    assert L.ptb_scene_create_from_device(dev.handle, tb._h, 1 << 28, mb._h, len(m), None, C.byref(h)) == -1
    assert b"2^28" in L.ptb_last_error() and not h.value
    # one below the limit is refused for the buffer size instead
    assert L.ptb_scene_create_from_device(dev.handle, tb._h, (1 << 28) - 1, mb._h, len(m), None, C.byref(h)) == -1
    assert b"tris buffer too small" in L.ptb_last_error()
    tb.close(); mb.close()


@pytest.mark.gpu
def test_arguments_are_checked(dev, pt, cornell):
    tris, mats = cornell
    L = pt.lib()
    n, nm = len(tris), len(mats)
    tb, mb = _upload(dev, tris), _upload(dev, mats)
    h = C.c_void_p()
    dh = dev.handle

    def refused(args, msg):
        assert L.ptb_scene_create_from_device(*args) == -1, msg
        assert msg in L.ptb_last_error(), (msg, L.ptb_last_error())
        assert not h.value

    for args in ((None, tb._h, n, mb._h, nm, None, C.byref(h)), (dh, None, n, mb._h, nm, None, C.byref(h)),
                 (dh, tb._h, n, None, nm, None, C.byref(h)), (dh, tb._h, n, mb._h, nm, None, None)):
        refused(args, b"null")
    for nt, nm_ in ((1, nm), (0, nm), (-5, nm), (n, 0), (n, -1)):
        refused((dh, tb._h, nt, mb._h, nm_, None, C.byref(h)), b"needs >= 2 triangles and >= 1 material")
    short_t, short_m = dev.buffer(n * 64 - 1), dev.buffer(nm * 64 - 16)
    refused((dh, short_t._h, n, mb._h, nm, None, C.byref(h)), b"tris buffer too small")
    refused((dh, tb._h, n, short_m._h, nm, None, C.byref(h)), b"mats buffer too small")
    # records 4 bytes into an allocation
    big = dev.buffer(n * 64 + 64)
    off_t = dev.wrap(big.device_ptr() + 4, n * 64)
    off_m = dev.wrap(big.device_ptr() + 4, nm * 64)
    refused((dh, off_t._h, n, mb._h, nm, None, C.byref(h)), b"16-byte aligned")
    refused((dh, tb._h, n, off_m._h, nm, None, C.byref(h)), b"16-byte aligned")
    for fw in (1, 3, 4, -1):
        refused((dh, tb._h, n, mb._h, nm, C.byref(pt.bvh_params(force_width=fw)), C.byref(h)), b"force_width")
    for pad in (0.0, -1e-4, float("nan"), float("inf")):
        refused((dh, tb._h, n, mb._h, nm, C.byref(pt.bvh_params(pad_rel=pad)), C.byref(h)), b"pad_rel must be a finite number > 0")
    ref = dev.scene(tris, mats, gpu_build=True)
    for fw in (0, 2):
        sc = dev.scene_from_device(tb, mb, pt.bvh_params(force_width=fw))
        assert_same_scene(ref, sc)
        sc.close()
    # buffers of another ptb_device (the same GPU) are refused
    other = pt.Device(0)
    ot = _upload(other, tris)
    refused((dh, ot._h, n, mb._h, nm, None, C.byref(h)), b"another device")
    refused((dh, tb._h, n, ot._h, nm, None, C.byref(h)), b"another device")
    ot.close(); other.close()
    for b in (short_t, short_m, off_t, off_m, big, tb, mb):
        b.close()
    ref.close()


@pytest.mark.gpu
def test_buffer_on_another_gpu_is_refused(dev, pt, cornell):
    count = C.c_int()
    pt.lib().ptb_device_count(C.byref(count))
    if count.value < 2:
        pytest.skip("needs two GPUs")
    tris, mats = cornell
    other = pt.Device(1)
    try:
        tb, mb = _upload(other, tris), _upload(dev, mats)
        with pytest.raises(pt.PtbError, match="another device"):
            dev.scene_from_device(tb, mb)
        tb.close(); mb.close()
    finally:
        other.close()


def _records(arr):
    return np.ascontiguousarray(arr).view(np.float32).reshape(-1, 16)


def _path_frame(dev, pt, sc):
    prm = pt.default_params(width=64, height=48, n_frames=2, mode=pt.MODE_PATH, accum=pt.ACCUM_LINEAR, max_depth=6, collect_stats=1)
    fb, sb = dev.buffer(64 * 48 * 16), dev.buffer(64 * 48 * 32)
    ctr = dev.render(sc, prm, fb, sb, want_counters=True)
    out = (fb.read(np.uint32).tobytes(), sb.read(np.uint8).tobytes(), ctr)
    fb.close(); sb.close()
    return out


@pytest.mark.gpu
def test_torch_tensors(pt, cornell):
    torch = pytest.importorskip("torch")
    tris, mats = cornell
    tess = pt.tessellate(tris, 20)
    src = torch.from_numpy(_records(tess)).cuda()
    mats_t = torch.from_numpy(_records(mats)).cuda()
    torch.cuda.synchronize()
    dev = pt.Device(0, stream=torch.cuda.current_stream().cuda_stream)
    try:
        ref = dev.scene(tess, mats, gpu_build=True)
        want = _path_frame(dev, pt, ref)
        # records written by torch on the current stream just before the call, behind a long kernel, with no synchronise:
        # read any earlier and the NaNs would be refused
        x = torch.full_like(src, float("nan"))
        torch.cuda._sleep(200_000_000)
        x.copy_(src)
        sc = dev.scene_from_device(x, mats_t)
        assert_same_scene(ref, sc)
        # the scene owns its copies: overwriting the inputs changes nothing
        keep = mats_t.clone()
        x.fill_(float("nan"))
        mats_t.fill_(float("nan"))
        assert _path_frame(dev, pt, sc) == want
        sc.close()
        mats_t = keep
        # numpy materials go up through a temporary Buffer
        x.copy_(src)
        sc = dev.scene_from_device(x, mats)
        assert _path_frame(dev, pt, sc) == want
        sc.close()
        with pytest.raises(pt.PtbError, match="aligned"):
            flat = torch.zeros(16 * len(tess) + 16, dtype=torch.float32, device="cuda")
            dev.scene_from_device(flat[1:1 + 16 * len(tess)].view(-1, 16), mats)
        with pytest.raises(pt.PtbError, match=r"shape \(n, 16\)"):
            dev.scene_from_device(x.view(-1, 8), mats)
        with pytest.raises(pt.PtbError, match="4-byte"):
            dev.scene_from_device(x.double(), mats)
        # creating and destroying scenes leaks no device memory
        free0 = None
        for it in range(20):
            s = dev.scene_from_device(x, mats_t)
            s.close()
            if it == 1:
                free0 = dev.memory()[0]
        assert dev.memory()[0] >= free0 - (8 << 20)
        ref.close()
    finally:
        dev.close()
    # a Device with its own stream would race with the torch work that wrote the records: refused
    own = pt.Device(0)
    try:
        with pytest.raises(pt.PtbError, match="current_stream"):
            own.scene_from_device(src, mats_t)
    finally:
        own.close()
