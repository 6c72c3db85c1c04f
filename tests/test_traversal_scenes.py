"""Every traversal form on scenes and rays that are not the Cornell box, against brute force and a float64 reference.

DESIGN.md section 4, "BVH equivalence": traversal may only skip triangles the reference loop would reject.  The scenes here are
random soups, the same soup offset to 1e4 and scaled by 1e3, a thin rod, a planar scene, mixed triangle sizes, exact duplicates,
triangles that share one centroid and two triangles, at sizes that reach the FLAT, 4-wide and binary forms.
CPU: the product's host builder equals the oracle's builder byte for byte; the oracle walking each form equals the brute-force
loop bit for bit on rays from within 100 scene diagonals; where a plain float64 ray-triangle test and the fp32 loop agree on a
clear winner, every tree returns it; rays from 300, 3000 and 30000 scene diagonals stay inside the measured envelope.
GPU: Device.intersect and Device.trace equal the oracle walking its own tree of every form (LBVH included) bit for bit, the
far-ray envelope holds for the kernels, PATH samples on a soup equal tests/oracle_shade.c, and degenerate scenes build on the
device.
"""
import ctypes as C
import functools
import os
import shutil
import subprocess

import numpy as np
import pytest

from conftest import ROOT, assert_same_tree, bits

FIELDS = ("tri", "t", "u", "v", "visits", "tests")
HIT_FIELDS = ("tri", "t", "u", "v")
FAR_DIAGONALS = (300, 3000, 30000)


# ---- scenes ------------------------------------------------------------------------------------------

def _triangles(p1, p2, p3):
    from oracle import binding as ob

    t = np.zeros(len(p1), ob.TRIANGLE_DTYPE)
    for k, p in (("p1", p1), ("p2", p2), ("p3", p3)):
        t[k][:, :3] = np.asarray(p, np.float32)
    t["id"] = 0
    return t


def soup(n, seed, size=0.03):
    """n random triangles with centres in [-1, 1]^3, edges of about 2.5 x size"""
    rng = np.random.default_rng(seed)
    c = rng.uniform(-1, 1, (n, 3))
    return _triangles(*(c + rng.normal(size=(n, 3)) * size for _ in range(3)))


def offset_soup(n, seed):
    t = soup(n, seed)
    for k in ("p1", "p2", "p3"):
        t[k][:, :3] += np.float32(1e4)
    return t


def scaled_soup(n, seed):
    t = soup(n, seed)
    for k in ("p1", "p2", "p3"):
        t[k][:, :3] *= np.float32(1e3)
    return t


def rod(n, seed):
    """a rod 20 long and 0.1 thick: the pad (1e-4 x diagonal) is a fiftieth of its thickness"""
    rng = np.random.default_rng(seed)
    c = rng.uniform([-10, -0.05, -0.05], [10, 0.05, 0.05], (n, 3))
    return _triangles(*(c + rng.normal(size=(n, 3)) * 0.01 for _ in range(3)))


def planar(n, seed):
    """every vertex at z = 0: zero scene extent on one axis"""
    t = soup(n, seed)
    for k in ("p1", "p2", "p3"):
        t[k][:, 2] = 0.0
    return t


def mixed(n, seed):
    """most triangles tiny, a few spanning half the scene"""
    rng = np.random.default_rng(seed)
    c = rng.uniform(-1, 1, (n, 3))
    size = np.where(rng.uniform(size=(n, 1)) < 0.05, 0.5, 0.005)
    return _triangles(*(c + rng.normal(size=(n, 3)) * size for _ in range(3)))


def duplicated(n, seed):
    """n/2 triangles, then the same records again in reverse order: every hit is a tie at equal t"""
    base = soup(n // 2, seed, size=0.06)
    return np.concatenate([base, base[::-1]])


def same_centroid(n, seed):
    """n different triangles that all have the box centre 0: p2 = -p1 and p3 inside that box"""
    rng = np.random.default_rng(seed)
    a = rng.uniform(0.2, 1.0, (n, 3)) * rng.choice([-1.0, 1.0], (n, 3))
    a = a.astype(np.float32)
    b = (rng.uniform(-1, 1, (n, 3)) * np.abs(a)).astype(np.float32)
    return _triangles(a, -a, b)


def two_triangles(n, seed):
    """the LBVH minimum"""
    return soup(2, seed, size=0.3)


KINDS = {"soup": soup, "offset": offset_soup, "scaled": scaled_soup, "rod": rod, "planar": planar, "mixed": mixed,
         "dup": duplicated, "centroid": same_centroid}
# 32 triangles: FLAT (at most 32 leaves whatever the SAH does); 256: 4-wide (fits 32 KB); 2000 / 3000: binary only
SCENES = {f"{k}-{n}": (k, n) for n in (32, 256, 2000) for k in KINDS}
SCENES["soup-3000"] = ("soup", 3000)
SCENES["two-2"] = ("two", 2)


@functools.lru_cache(maxsize=None)
def scene(name):
    kind, n = SCENES[name]
    seed = 1000 + sorted(SCENES).index(name)
    return (two_triangles if kind == "two" else KINDS[kind])(n, seed)


def forms(ob, tris):
    """the forms the product can build for this scene (ptb_scene_create with force_width): FLAT when the oracle's FLAT build
    succeeds, 4-wide when its 4-wide nodes, triangles and material fit 32 KB, binary always"""
    out = []
    if len(tris) <= 64:
        try:
            ob.build_bvh(tris, width=1)
            out.append(1)
        except RuntimeError:
            pass
    if len(tris) <= 2048:
        b4 = ob.build_bvh(tris, width=4)
        if len(b4["nodes"]) * 128 + len(tris) * 48 + 32 <= 32 * 1024 and b4["bfs_nodes"] == len(b4["nodes"]):
            out.append(4)
    return out + [2]


def bounds(tris):
    v = np.concatenate([tris[k][:, :3] for k in ("p1", "p2", "p3")]).astype(np.float64)
    lo, hi = v.min(0), v.max(0)
    return lo, hi, (lo + hi) / 2, float(np.linalg.norm(hi - lo))


# ---- rays --------------------------------------------------------------------------------------------

def _points_on_triangles(rng, tris, n):
    """a random interior point of a random triangle, per ray"""
    i = rng.integers(0, len(tris), n)
    w = rng.dirichlet([1, 1, 1], n)
    return sum(w[:, k:k + 1] * tris[f][i, :3].astype(np.float64) for k, f in enumerate(("p1", "p2", "p3")))


def _unit(v):
    return (v / np.linalg.norm(v, axis=1, keepdims=True)).astype(np.float32)


def near_rays(tris, n, seed):
    """origins within 100 scene diagonals: a quarter inside the scene's box in random directions, a quarter inside it aimed at
    the triangles, a third on spheres of 0.5 to 100 diagonals aimed at the triangles, the rest axis-parallel through them"""
    rng = np.random.default_rng(seed)
    lo, hi, ctr, diag = bounds(tris)
    slack = 0.1 * diag
    o = rng.uniform(lo - slack, hi + slack, (n, 3))
    tgt = _points_on_triangles(rng, tris, n)
    d = tgt - o
    q = n // 4
    d[:q] = rng.normal(size=(q, 3))
    far = slice(2 * q, 2 * q + n // 3)
    m = far.stop - far.start
    s = rng.normal(size=(m, 3))
    s /= np.linalg.norm(s, axis=1, keepdims=True)
    o[far] = ctr + s * (diag * np.exp(rng.uniform(np.log(0.5), np.log(100.0), (m, 1))))
    d[far] = tgt[far] - o[far]
    ax = slice(far.stop, n)
    m = n - far.stop
    axis, sign = rng.integers(0, 3, m), rng.choice([-1.0, 1.0], m)
    dd = np.zeros((m, 3))
    dd[np.arange(m), axis] = sign
    d[ax] = dd
    o[ax] = tgt[ax] - dd * rng.uniform(0.05, 2.0, (m, 1)) * diag
    return o.astype(np.float32), _unit(d)


def far_rays(tris, n, diagonals, seed):
    """origins on a sphere of `diagonals` scene diagonals around the scene's centre, each aimed at a point on a triangle"""
    rng = np.random.default_rng(seed)
    _lo, _hi, ctr, diag = bounds(tris)
    s = rng.normal(size=(n, 3))
    o = ctr + s / np.linalg.norm(s, axis=1, keepdims=True) * (diagonals * diag)
    return o.astype(np.float32), _unit(_points_on_triangles(rng, tris, n) - o)


def _tmax_mix(rng, hit_t, n, scale):
    """per-ray tmax from {1e20, random, exactly the closest hit's t (strict <: a miss), 0, negative, NaN}, as tests/test_intersect.py"""
    kind = rng.integers(0, 6, n)
    tm = np.full(n, 1e20, np.float32)
    tm[kind == 1] = rng.uniform(0.0, scale, (kind == 1).sum()).astype(np.float32)
    exact = (kind == 2) & (hit_t > 0)
    tm[exact] = hit_t[exact]
    tm[kind == 3] = 0.0
    tm[kind == 4] = -rng.uniform(0.0, scale, (kind == 4).sum()).astype(np.float32)
    tm[kind == 5] = np.nan
    return tm, exact


# ---- the float64 reference ---------------------------------------------------------------------------

def mt64(tris, o, d, idx=None):
    """one-sided Moller-Trumbore in float64 on the fp32 vertices (det > 0, as the reference's det >= 1e-8).
    idx None: every triangle for every ray -> (det, u, v, t) of shape (n_rays, n_tris); else triangle idx[i] for ray i."""
    p = [tris[k][:, :3].astype(np.float64) for k in ("p1", "p2", "p3")]
    o, d = np.asarray(o, np.float64), np.asarray(d, np.float64)
    if idx is not None:
        p = [x[idx] for x in p]
    else:
        p = [x[None] for x in p]
        o, d = o[:, None], d[:, None]
    e1, e2 = p[1] - p[0], p[2] - p[0]
    pv = np.cross(d, e2)
    det = (e1 * pv).sum(-1)
    with np.errstate(divide="ignore", invalid="ignore"):
        tv = o - p[0]
        u = (tv * pv).sum(-1) / det
        qv = np.cross(tv, e1)
        v = (d * qv).sum(-1) / det
        t = (e2 * qv).sum(-1) / det
    return det, u, v, t


def crosses64(tris, o, d, tri):
    """float64: ray i truly crosses triangle tri[i] (det > 0, barycentrics in [0, 1], t > 0); False where tri < 0"""
    ok = tri >= 0
    det, u, v, t = mt64(tris, o, d, np.where(ok, tri, 0))
    with np.errstate(invalid="ignore"):
        return ok & (det > 0) & (u >= 0) & (v >= 0) & (u + v <= 1) & (t > 0)


def clear_winner64(tris, o, d, chunk=256):
    """per ray: the triangle the float64 test hits first when that hit is clear -- its barycentrics are all >= 1e-3 and every
    other float64 hit is farther by a relative 1e-4 in t -- else -1.  Exact copies of a triangle are one hit, and the lowest
    index wins it, as in the reference loop."""
    verts = np.ascontiguousarray(np.stack([tris[k][:, :3] for k in ("p1", "p2", "p3")], 1)).view(np.uint8).reshape(len(tris), -1)
    _u, first, inverse = np.unique(verts, axis=0, return_index=True, return_inverse=True)
    copy_of = first[inverse.ravel()]  # the lowest index with the same three vertices
    out = np.full(len(o), -1, np.int32)
    for s in range(0, len(o), chunk):
        det, u, v, t = mt64(tris, o[s:s + chunk], d[s:s + chunk])
        with np.errstate(invalid="ignore"):
            hit = (det > 0) & (u >= 0) & (v >= 0) & (u + v <= 1) & (t > 0)
            tt = np.where(hit, t, np.inf)
            best = np.argmin(tt, axis=1)
            r = np.arange(len(best))
            t1 = tt[r, best]
            t2 = np.where(copy_of[None, :] != copy_of[best][:, None], tt, np.inf).min(axis=1)
            b = best
            clear = np.isfinite(t1) & (np.minimum(np.minimum(u[r, b], v[r, b]), 1 - u[r, b] - v[r, b]) >= 1e-3) & (t2 > t1 * (1 + 1e-4))
        out[s:s + chunk] = np.where(clear, best, -1)
    return out


# ---- oracle helpers ----------------------------------------------------------------------------------

def _oracle_ext(tmp_path_factory, src, name):
    """tests/<src> compiled with the compiler and flags of oracle/Makefile, together with the oracle's builder"""
    out = tmp_path_factory.mktemp(name) / f"lib{name}.so"
    cc = shutil.which("gcc", path="/usr/bin") or "gcc"
    subprocess.check_call([cc, "-O2", "-std=c11", "-fPIC", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-fno-math-errno",
                           "-mfma", "-shared", "-I", os.path.join(ROOT, "oracle"), "-o", str(out),
                           os.path.join(ROOT, "tests", src), os.path.join(ROOT, "oracle", "oracle_bvh.c"), "-lm"])
    return C.CDLL(str(out))


@pytest.fixture(scope="module")
def closest_tmax(ob, tmp_path_factory):
    """closest_tmax(tris, o, d, tmax, bvh) -> dict like ob.trace's: the oracle's closest-hit query with a per-ray tmax
    (tests/oracle_tmax.c)"""
    lib = _oracle_ext(tmp_path_factory, "oracle_tmax.c", "oracle_tmax")
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


def oracle_form(ob, tris, form, **params):
    """(ora_bvh, keepalive, built dict) of the oracle's own tree; form 1 | 4 | 2 (quantised, as the product walks it) or
    "2f" (the binary tree on its fp32 boxes: the boxes the FLAT and 4-wide forms are made of)"""
    b = ob.build_bvh(tris, ob.bvh_params(**params) if params else None, width=2 if form == "2f" else form)
    bvh, keep = ob.make_bvh(b["nodes"], b["tri_order"], quantized=form != "2f")
    return bvh, keep, b


@functools.lru_cache(maxsize=None)
def _brute(name, which, n, seed):
    """the brute-force loop's closest hits (tmax 1e20) on a scene's near or far rays, computed once per module run"""
    from oracle import binding as ob

    tris = scene(name)
    o, d = near_rays(tris, n, seed) if which == "near" else far_rays(tris, n, which, seed)
    return o, d, ob.trace(tris, o, d, np.float32(1e20))


def _mismatch(a, b):
    return (a["tri"] != b["tri"]) | (bits(a["t"]) != bits(b["t"])) | (bits(a["u"]) != bits(b["u"])) | (bits(a["v"]) != bits(b["v"]))


N_NEAR = 40_000


# ---- no device needed --------------------------------------------------------------------------------

@pytest.mark.parametrize("name", sorted(SCENES))
def test_host_builder_equals_the_oracles_builder(pt, ob, name):
    tris = scene(name)
    fs = forms(ob, tris)
    assert fs == {32: [1, 4, 2], 256: [4, 2]}.get(len(tris), [1, 4, 2] if len(tris) == 2 else [2]), fs
    for form in fs:
        p, o = pt.build_bvh_host(tris, width=form), ob.build_bvh(tris, width=form)
        assert_same_tree(p["nodes"], p["tri_order"], o)
        assert p["depth"] == o["depth"], form


@pytest.mark.parametrize("name", sorted(SCENES))
def test_every_form_equals_brute_force_on_near_rays(ob, closest_tmax, name):
    """closest hit: triangle and the bits of t, u, v; any hit: hit or miss -- at tmax 1e20 and at the tmax mix"""
    tris = scene(name)
    o, d, br = _brute(name, "near", N_NEAR, 7)
    assert (br["tri"] >= 0).mean() > 0.3
    tm, exact = _tmax_mix(np.random.default_rng(8), br["t"], len(o), 2 * bounds(tris)[3])
    br_tm = closest_tmax(tris, o, d, tm)
    br_any = ob.trace(tris, o, d, tm, any_hit=True)
    assert ((br_tm["tri"] >= 0) == (br_any["tri"] >= 0)).all()
    for form in forms(ob, tris) + ["2f"]:
        bvh, _keep, _b = oracle_form(ob, tris, form)
        g = ob.trace(tris, o, d, np.float32(1e20), bvh=bvh)
        bad = _mismatch(g, br)
        assert not bad.any(), f"{name} form {form}: {bad.sum()} of {len(o)} rays differ from brute force, e.g. ray {np.flatnonzero(bad)[:5]}"
        g = closest_tmax(tris, o, d, tm, bvh)
        assert not _mismatch(g, br_tm).any(), f"{name} form {form}: closest hit with the tmax mix"
        assert (g["tri"][exact] == -1).all()
        g = ob.trace(tris, o, d, tm, bvh=bvh, any_hit=True)
        np.testing.assert_array_equal(g["tri"] >= 0, br_any["tri"] >= 0, err_msg=f"{name} form {form}: any hit")


SMALLEST_PAD_REL = 1e-5  # include/ptb200.h, ptb_bvh_params.pad_rel


def test_near_ray_equivalence_holds_down_to_the_documented_pad_rel(ob):
    """the smallest pad_rel include/ptb200.h documents keeps every form equal to brute force on every scene's near rays; at 3e-6
    the planar scenes lose hits on their fp32 boxes"""
    for name in sorted(SCENES):
        tris = scene(name)
        o, d, br = _brute(name, "near", N_NEAR, 7)
        for form in forms(ob, tris) + ["2f"]:
            bvh, _keep, _b = oracle_form(ob, tris, form, pad_rel=SMALLEST_PAD_REL)
            bad = _mismatch(ob.trace(tris, o, d, np.float32(1e20), bvh=bvh), br)
            assert not bad.any(), f"{name} form {form}: {bad.sum()} rays differ from brute force at pad_rel {SMALLEST_PAD_REL}"


@pytest.mark.parametrize("name", sorted(SCENES))
def test_every_form_returns_the_float64_clear_winner(ob, name):
    """where a plain float64 test and the fp32 loop agree on a clear winner, every tree returns it; the two agree almost always"""
    tris = scene(name)
    o, d, br = _brute(name, "near", N_NEAR, 7)
    k = slice(0, None, 10 if len(tris) > 1000 else 4)  # every kind of near ray, spread over the generator's parts
    o, d, br = o[k], d[k], {f: a[k] for f, a in br.items()}
    win = clear_winner64(tris, o, d)
    agree = (win >= 0) & (br["tri"] == win)
    assert (win >= 0).sum() > 0.1 * len(o), name
    # fp32 barycentrics are off by about |o| 2^-24 / edge: on the rod's small triangles seen from 100 diagonals that can exceed
    # the 1e-3 margin, so a few rays in a thousand may disagree there
    assert agree.sum() >= 0.99 * (win >= 0).sum(), f"{name}: the fp32 loop disagrees with a clear float64 winner"
    for form in forms(ob, tris) + ["2f"]:
        bvh, _keep, _b = oracle_form(ob, tris, form)
        g = ob.trace(tris, o, d, np.float32(1e20), bvh=bvh)
        lost = agree & (g["tri"] != win)
        assert not lost.any(), f"{name} form {form}: {lost.sum()} clear hits lost, e.g. ray {np.flatnonzero(lost)[:5]}"


def far_ray_envelope(tris, o, d, br, g):
    """(mismatches, unexplained): a mismatch is explained when the tree's t is within 2^-16 t of brute force's, or when brute
    force's triangle fails the float64 test"""
    bad = _mismatch(g, br)
    close = (g["tri"] >= 0) & (np.abs(g["t"].astype(np.float64) - br["t"]) <= br["t"].astype(np.float64) * 2.0 ** -16)
    unexplained = bad & ~close & crosses64(tris, o, d, np.where(bad, br["tri"], -1))
    return int(bad.sum()), int(unexplained.sum())


FAR_BOUND = {300: 1e-5, 3000: 1e-3, 30000: 2e-2}  # mismatch rate; unexplained mismatches: none up to 3000 diagonals
N_FAR = 400_000


@pytest.mark.parametrize("diagonals", FAR_DIAGONALS)
@pytest.mark.parametrize("name", ["soup-3000", "soup-256", "soup-32"])
def test_far_rays_stay_inside_the_envelope(ob, name, diagonals):
    """DESIGN.md section 4: origins hundreds of scene diagonals away break the equivalence, by the best_t cull (Moller-Trumbore's
    t is off by more than the pad along the ray) and by the rounding of o * invd in the slab test"""
    tris = scene(name)
    o, d, br = _brute(name, diagonals, N_FAR, 11)
    assert (br["tri"] >= 0).mean() > 0.25  # one-sided triangles: a ray aimed at a back face passes
    for form in forms(ob, tris) + ["2f"]:
        bvh, _keep, _b = oracle_form(ob, tris, form)
        bad, unexplained = far_ray_envelope(tris, o, d, br, ob.trace(tris, o, d, np.float32(1e20), bvh=bvh))
        print(f"{name} form {form} at {diagonals} diagonals: {bad} of {len(o)} rays differ from brute force, {unexplained} unexplained")
        assert bad <= FAR_BOUND[diagonals] * len(o), (form, bad)
        if diagonals <= 3000:
            assert unexplained == 0, (form, unexplained)


@pytest.mark.parametrize("pad_rel", [0.0, -1e-4, float("nan"), float("inf")])
def test_pad_rel_must_be_a_positive_number(pt, pad_rel):
    with pytest.raises(pt.PtbError, match="pad_rel"):
        pt.build_bvh_host(soup(40, 1), pt.bvh_params(pad_rel=pad_rel), width=2)


# ---- on the B200 -------------------------------------------------------------------------------------

def _pack(o, d, tmax):
    r = np.zeros((len(o), 8), np.float32)
    r[:, 0:3], r[:, 3], r[:, 4:7] = o, tmax, d
    return r


def _intersect(dev, sc, o, d, tmax, any_hit):
    n = len(o)
    rb, hb, sb = dev.buffer(n * 32), dev.buffer(n * 16), dev.buffer(n * 8)
    rb.write(_pack(o, d, tmax))
    dev.intersect(sc, rb, hb, any_hit=any_hit, stats=sb)
    h = hb.read(np.uint8, count=n * 16).view(np.float32).reshape(-1, 4)
    s = sb.read(np.uint32, count=2 * n).reshape(-1, 2)
    for b in (rb, hb, sb):
        b.close()
    return {"tri": h[:, 3].view(np.int32).copy(), "t": h[:, 0].copy(), "u": h[:, 1].copy(), "v": h[:, 2].copy(),
            "visits": s[:, 0].copy(), "tests": s[:, 1].copy()}


def _gpu_rays(tris, seed):
    """near rays and far rays from every distance of the envelope"""
    parts = [near_rays(tris, 24_000, seed)] + [far_rays(tris, 4000, r, seed + r) for r in FAR_DIAGONALS]
    return np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts])


def _product_scene(dev, pt, mats, tris, form):
    if form == "lbvh":
        return dev.scene(tris, mats, gpu_build=True)
    return dev.scene(tris, mats, pt.bvh_params(force_width=form))


@pytest.fixture(scope="module")
def one_material(pt):
    m = np.zeros(1, pt.MATERIAL_DTYPE)
    m["albedo"] = [0.7, 0.7, 0.7, 1.0]
    m["emissive"] = [0.0, 0.0, 0.0, 1.0]
    m["type"] = 1
    return m


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(SCENES))
def test_intersect_and_trace_equal_the_oracle(dev, pt, ob, closest_tmax, one_material, name):
    """every form the scene qualifies for, and its LBVH: tri, t, u, v, node visits and triangle tests of Device.intersect
    (closest and any hit at the tmax mix) and Device.trace (closest at 1e20, any at the tmax mix) == the oracle on its own tree;
    binary trees with the traversal stack in local and in shared memory"""
    tris = scene(name)
    o, d = _gpu_rays(tris, 21)
    for form in forms(ob, tris) + ["lbvh"]:
        sc = _product_scene(dev, pt, one_material, tris, form)
        try:
            width = sc.info()["width"]
            if form == "lbvh":
                assert width == 2
                bvh, _keep = ob.make_bvh(*sc.bvh())
            else:
                assert width == form
                bvh, _keep, ob_ = oracle_form(ob, tris, form)
                assert_same_tree(*sc.bvh(), ob_)
            ref = ob.trace(tris, o, d, np.float32(1e20), bvh=bvh)
            tm, exact = _tmax_mix(np.random.default_rng(22), ref["t"], len(o), 2 * bounds(tris)[3])
            want = {False: closest_tmax(tris, o, d, tm, bvh), True: ob.trace(tris, o, d, tm, bvh=bvh, any_hit=True)}
            for stack in ((0, 2) if width == 2 else (0,)):
                dev.set_tuning(2, stack)
                try:
                    for any_hit in (False, True):
                        msg = f"{name} {form} stack={stack} any={any_hit}"
                        got = _intersect(dev, sc, o, d, tm, any_hit)
                        for f in HIT_FIELDS:
                            np.testing.assert_array_equal(bits(got[f]), bits(want[any_hit][f]), err_msg=f"{msg} {f}")
                        # any-hit rays with a NaN tmax on binary trees: the oracle's pop drops deferred entries (DESIGN.md
                        # section 4, tests/test_intersect.py); both report a miss
                        cmp = ~np.isnan(tm) if (any_hit and width == 2) else np.ones(len(o), bool)
                        for f in ("visits", "tests"):
                            np.testing.assert_array_equal(got[f][cmp], want[any_hit][f][cmp], err_msg=f"{msg} {f}")
                        assert (got["tri"][exact] == -1).all()
                    got = dev.trace(sc, o, d, np.float32(1e20))
                    for f in FIELDS:
                        np.testing.assert_array_equal(bits(got[f]), bits(ref[f]), err_msg=f"{name} {form} stack={stack} trace {f}")
                    got = dev.trace(sc, o, d, tm, any_hit=True)
                    for f in HIT_FIELDS:
                        np.testing.assert_array_equal(bits(got[f]), bits(want[True][f]), err_msg=f"{name} {form} trace any {f}")
                finally:
                    dev.set_tuning(2, 0)
        finally:
            sc.close()


@pytest.mark.gpu
@pytest.mark.parametrize("diagonals", FAR_DIAGONALS)
def test_far_rays_stay_inside_the_envelope_on_the_device(dev, pt, ob, one_material, diagonals):
    """the kernels' brute-force loop equals the oracle's bit for bit, and the kernels' trees keep the CPU envelope"""
    for name in ("soup-3000", "soup-256", "soup-32"):
        tris = scene(name)
        o, d, br = _brute(name, diagonals, N_FAR, 11)
        for form in forms(ob, tris) + ["lbvh"]:
            sc = _product_scene(dev, pt, one_material, tris, form)
            try:
                gbr = dev.trace(sc, o, d, np.float32(1e20), accel=pt.ACCEL_BRUTE)
                assert not _mismatch(gbr, br).any(), f"{name}: the device's brute-force loop differs from the oracle's"
                bad, unexplained = far_ray_envelope(tris, o, d, br, _intersect(dev, sc, o, d, np.full(len(o), 1e20, np.float32), False))
                print(f"device {name} {form} at {diagonals} diagonals: {bad} of {len(o)} differ, {unexplained} unexplained")
                assert bad <= FAR_BOUND[diagonals] * len(o), (name, form, bad)
                if diagonals <= 3000:
                    assert unexplained == 0, (name, form, unexplained)
            finally:
                sc.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["two-2", "centroid-32", "centroid-256", "centroid-2000"])
def test_degenerate_scenes_build_on_the_device(dev, pt, ob, one_material, name):
    """two triangles (the LBVH minimum) and triangles with one shared centroid (every Morton code equal): built by
    ptb_scene_create_gpu, their hits equal brute force's on near rays"""
    tris = scene(name)
    o, d, br = _brute(name, "near", N_NEAR, 7)
    sc = dev.scene(tris, one_material, gpu_build=True)
    try:
        assert sc.info()["width"] == 2 and sc.info()["n_nodes"] == len(tris) - 1
        got = _intersect(dev, sc, o, d, np.full(len(o), 1e20, np.float32), False)
        assert not _mismatch(got, br).any(), name
        got = _intersect(dev, sc, o, d, np.full(len(o), 1e20, np.float32), True)
        np.testing.assert_array_equal(got["tri"] >= 0, br["tri"] >= 0)
    finally:
        sc.close()


@pytest.mark.gpu
@pytest.mark.parametrize("gpu_build", [False, True])
def test_scene_create_refuses_pad_rel_that_is_not_positive(dev, pt, one_material, gpu_build):
    for pad_rel in (0.0, -1e-4, float("nan"), float("inf")):
        with pytest.raises(pt.PtbError, match="pad_rel"):
            dev.scene(soup(256, 2), one_material, pt.bvh_params(pad_rel=pad_rel), gpu_build=gpu_build)


@pytest.fixture(scope="module")
def ora_shade(ob, tmp_path_factory):
    """ora_shade(prm, tris, mats, o, d, seeds, bvh) -> (float4 per ray, stats per ray, counters dict) (tests/oracle_shade.c)"""
    lib = _oracle_ext(tmp_path_factory, "oracle_shade.c", "oracle_shade")
    lib.ora_shade.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int] + [C.c_void_p] * 6

    def run(prm, tris, mats, o, d, seeds, bvh):
        n = len(o)
        prm.use_bvh = 1
        tris, mats = np.ascontiguousarray(tris), np.ascontiguousarray(mats)
        o, d = np.ascontiguousarray(o, np.float32), np.ascontiguousarray(d, np.float32)
        seeds = np.ascontiguousarray(seeds, np.uint32)
        rad, st, ctr = np.zeros((n, 4), np.float32), np.zeros(n, ob.STATS_DTYPE), ob.Counters()
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        assert lib.ora_shade(C.byref(prm), p(tris), len(tris), p(mats), C.cast(C.byref(bvh), C.c_void_p), n, p(o), p(d),
                             p(seeds), p(rad), p(st), C.byref(ctr)) == 0
        return rad, st, ctr.as_dict()

    return run


@pytest.mark.gpu
def test_shade_path_on_a_soup_equals_the_oracle(dev, pt, ob, cornell, ora_shade):
    """PATH samples on a 2000-triangle soup (binary form) lit by a quad made of two of its triangles: radiance, statistics and
    counters == tests/oracle_shade.c on the oracle's own tree"""
    _tris, cmats = cornell
    tris = scene("soup-2000").copy()
    mats = cmats[[0, 5, 8]]  # diffuse grey, the Cornell light, glossy
    tris["id"][::7] = 2
    a, ea, eb = np.float32([-0.3, 1.3, -0.3]), np.float32([0.6, 0, 0]), np.float32([0, 0, 0.6])
    for k, (p1, p2, p3) in enumerate(((a, a + ea, a + ea + eb), (a, a + eb, a + ea + eb))):
        tris["p1"][10 + k, :3], tris["p2"][10 + k, :3], tris["p3"][10 + k, :3] = p1, p2, p3
        tris["id"][10 + k] = 1
    p1, lea, leb = ob.light_from_quad(tris, 1)
    assert np.allclose(lea, ea) and np.allclose(leb, eb)
    rng = np.random.default_rng(90)
    o, d = near_rays(tris, 20_000, 91)
    seeds = rng.integers(0, 1 << 32, len(o), dtype=np.uint64).astype(np.uint32)
    sc = dev.scene(tris, mats)
    try:
        assert sc.info()["width"] == 2
        bvh, _keep, b = oracle_form(ob, tris, 2)
        assert_same_tree(*sc.bvh(), b)
        prm = pt.default_params(mode=pt.MODE_PATH, max_depth=6, light_quad=1, light_p1=p1, light_ea=lea, light_eb=leb)
        oprm = ob.default_params(1, 1, mode=ob.MODE_PATH, max_depth=6, light_quad=1, light_p1=p1, light_ea=lea, light_eb=leb)
        rb, radb, sb = dev.buffer(len(o) * 32), dev.buffer(len(o) * 16), dev.buffer(len(o) * 32)
        r = np.zeros(len(o), pt.SAMPLE_RAY_DTYPE)
        r["o"], r["seed"], r["d"] = o, seeds, d
        rb.write(r)
        _, ctr = dev.shade(sc, prm, rb, radb, stats=sb, want_counters=True)
        rad, st = radb.read(np.float32, count=4 * len(o)).reshape(-1, 4), sb.read(pt.STATS_DTYPE, count=len(o))
        for x in (rb, radb, sb):
            x.close()
        want_rad, want_st, want_ctr = ora_shade(oprm, tris, mats, o, d, seeds, bvh)
        np.testing.assert_array_equal(bits(rad), bits(want_rad))
        assert st.tobytes() == want_st.tobytes()
        for f in ("rays_closest", "rays_any", "nodes", "tri_tests", "samples"):
            assert ctr[f] == want_ctr[f], f
        assert (st["tri"] >= 0).mean() > 0.3 and (rad[:, :3] > 0).any()
    finally:
        sc.close()
