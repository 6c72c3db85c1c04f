"""The render modes on materials and lights the Cornell box never uses: the kernels against the oracle bit for bit, and the
shading of both against float64 restatements of DESIGN.md section 4.

Part A (GPU): material tables for the Cornell geometry with diffuse albedo 0 to 1.5 and up to 1e25 (masks that overflow), GGX roughness 0 to 2, material types
the BSDF does not know (0, 3, -1, a NaN bit pattern), emission on several quads (coloured, on a specular quad, -0.0, one
negative component) and garbage in albedo.w, emissive.w and the padding; DIRECT lights other than quad 5, outside the quad
list, tilted away from part of the box and degenerate; the FLAT (auto and 64 triangles in 32 leaves), 4-wide and binary
forms (shared-memory stack and LBVH too), and a scene whose normals straddle the 0.001 tangent-frame threshold.  ptb_render
(megakernel and wavefront, BVH and brute force) and ptb_scene_shade equal the oracle on its own tree: radiance bits (NaN at
the same positions; payloads are outside the contract, DESIGN.md section 2), statistics and counters.
Part B (CPU on the oracle, GPU on the kernels): a diffuse furnace whose samples must be the float64 geometric sums, DIRECT's
mean under a parallelogram light against Lambert's form factor and float64 quadrature, fully shadowed points, and per-sample
DIRECT and AO on a floor under occluders against a float64 restatement with the same integer RNG draws, on the samples whose
float64 decisions all have a clear margin.
"""
import numpy as np
import pytest

from conftest import bits, oracle_tree
from test_shade import _odd_rays, _shade, ora_shade  # noqa: F401  (ora_shade is a fixture)
from test_traversal_scenes import _triangles, clear_winner64, mt64

NAN_TYPE = 0x7FA00000  # a signalling-NaN bit pattern in the float lane the device packs `type` into


# ---- material tables for the Cornell geometry ------------------------------------------------------
# quads: 0 ceiling, 1 back wall, 2 floor, 3-4 box bottoms (hidden), 5 ceiling light, 6 right wall, 7 left wall,
# 8-12 short box, 13-17 tall box

def _material_table(ob, spec):
    """18 materials from {quad: (albedo, emissive, roughness, type)}; the rest diffuse grey.  albedo.w, emissive.w and the
    24 padding bytes hold garbage (NaN bit patterns, 0xFF), which must change nothing."""
    m = np.zeros(18, ob.MATERIAL_DTYPE)
    m["albedo"][:, :3] = 0.7
    m["type"] = 1
    for q, (alb, emi, rough, typ) in spec.items():
        m["albedo"][q, :3], m["emissive"][q, :3], m["roughness"][q], m["type"][q] = alb, emi, rough, typ
    raw = m.view(np.uint8).reshape(18, 64)
    raw[:, 12:16] = 0xFF
    raw[:, 28:32] = np.frombuffer(np.uint32(0x7FC00001).tobytes(), np.uint8)
    raw[:, 40:64] = 0xFF
    return m


def tables(ob):
    box = lambda qs, v: {q: v for q in qs}
    t = {}
    t["albedo"] = _material_table(ob, {
        0: ((0.7, 0.6, 0.5), (0.0, 0.5, 0.25), 0.0, 1),   # coloured emission with x = 0
        1: ((1.5, 1.0, 0.7), (0.0, 0.0, 0.0), 0.0, 1),
        2: ((3e19, 1.0, 1.0), (0.0, 0.0, 0.0), 0.0, 1),    # with the boxes: masks that overflow to inf
        5: ((0.7, 0.7, 0.7), (30.0, 20.0, 10.0), 0.0, 1),
        6: ((0.0, 0.0, 0.0), (0.3, -0.2, 0.1), 0.0, 1),   # one negative component
        7: ((0.2, 1.5, 0.4), (-0.0, -0.0, -0.0), 0.0, 1),
        **box(range(8, 13), ((1e25, 1.0, 0.25), (0.0, 0.0, 0.0), 0.0, 1)),
        **box(range(13, 18), ((0.9, 0.8, 0.7), (2.0, 1.0, 0.5), 0.3, 2)),  # emission on a specular quad
    })
    t["ggx"] = _material_table(ob, {
        0: ((0.7, 0.7, 0.7), (0.0, 0.0, 0.0), 2.0, 2),
        1: ((0.8, 0.7, 0.6), (0.0, 0.0, 0.0), 0.0, 2),     # roughness 0: the reference's GGX term is 0/0
        2: ((0.7, 0.7, 0.7), (0.0, 0.0, 0.0), 0.05, 2),
        5: ((0.7, 0.7, 0.7), (30.0, 30.0, 30.0), 0.0, 1),
        6: ((0.6, 0.2, 0.2), (0.0, 0.0, 0.0), 1e-3, 2),
        7: ((0.2, 0.6, 0.2), (0.0, 0.0, 0.0), 1.0, 2),
        **box(range(8, 13), ((0.5, 0.35, 0.05), (0.0, 0.0, 0.0), 0.3, 2)),
        **box(range(13, 18), ((0.5, 0.5, 0.5), (0.0, 0.0, 0.0), 0.0, 2)),
    })
    t["types"] = _material_table(ob, {
        0: ((0.7, 0.7, 0.7), (0.0, 0.0, 0.0), 0.3, 2),
        1: ((0.7, 0.7, 0.7), (0.0, 0.0, 0.0), 0.0, 0),
        2: ((0.7, 0.7, 0.7), (1.0, 2.0, 3.0), 0.0, 3),
        5: ((0.7, 0.7, 0.7), (30.0, 30.0, 30.0), 0.0, 1),
        6: ((0.6, 0.0, 0.0), (0.0, 0.0, 0.0), 0.0, -1),
        7: ((0.0, 0.6, 0.0), (0.0, 0.0, 0.0), 0.0, NAN_TYPE),
        **box(range(8, 13), ((0.5, 0.35, 0.05), (0.0, 0.0, 0.0), 0.008, NAN_TYPE)),
        **box(range(13, 18), ((0.7, 0.7, 0.7), (0.0, 0.0, 0.0), 0.0, 1)),
    })
    return t


UNKNOWN_TYPE_QUADS = (1, 2, 6, 7, 8, 9, 10, 11, 12)  # of tables()["types"]


def lights(ob, tris):
    """name -> (light_quad, p1, ea, eb, derive): derive = the device takes the light from the first triangle pair of light_quad
    in the scene `tris` (ea = 0), the oracle gets the same parallelogram explicitly"""
    L = {"quad5": (5, *ob.light_from_quad(tris, 5), True), "quad0": (0, *ob.light_from_quad(tris, 0), True)}
    L["outside"] = (5, [-1.0, 4.8, -1.6], [0.0, 0.0, -1.1], [1.3, 0.0, 0.0], False)  # faces down, in no quad
    L["tilted"] = (5, [0.0, 1.0, -1.5], [0.0, 2.0, 0.0], [0.0, 0.0, -2.0], False)    # faces -x: cos_l <= 0 for x > 0
    L["degenerate"] = (5, [-0.5, 5.3, -2.5], [1.0, 0.0, 0.0], [0.5, 0.0, 0.0], False)  # ea || eb
    return L


def _light_kw(light, device):
    q, p1, ea, eb, derive = light
    if device and derive:
        return dict(light_quad=q)
    return dict(light_quad=q, light_p1=p1, light_ea=ea, light_eb=eb)


def _mode_variants(ob, tris, names=None):
    """(mode, light name or None) pairs: every mode, DIRECT under each light"""
    out = [(0, None), (1, None), (3, None)]
    return out + [(2, n) for n in (names or lights(ob, tris))]


# ---- scenes ------------------------------------------------------------------------------------------

def _quads(corners, ids):
    """triangle pairs (p1, p2, p3), (p3, p4, p1) of each quad (p1, p2, p3, p4), as the scene format and tessellate expect"""
    c = np.asarray(corners, np.float64)
    t = _triangles(np.concatenate([c[:, 0], c[:, 2]]), np.concatenate([c[:, 1], c[:, 3]]), np.concatenate([c[:, 2], c[:, 0]]))
    t["id"] = np.concatenate([ids, ids])
    n = len(c)
    return t[np.stack([np.arange(n), np.arange(n) + n], 1).ravel()]


def flat_limit(cornell_tris):
    """the Cornell box plus 14 small quads inside it: 64 triangles in 32 FLAT leaves"""
    rng = np.random.default_rng(0)
    c = rng.uniform([-2.3, 0.4, -5.0], [2.3, 5.0, -0.6], (14, 3))
    a, b = rng.normal(size=(14, 3)) * 0.12, rng.normal(size=(14, 3)) * 0.12
    extra = _quads(np.stack([c, c + a, c + a + b, c + b], 1), np.arange(14) % 18)
    return np.concatenate([cornell_tris, extra])


def _facing_quads(corners, ids, d):
    """quads whose front faces rays along d[i] (the reference's test is one-sided: det >= 1e-8): corners reversed where not"""
    c = np.array(corners, np.float32)
    t = _quads(c, ids)[::2]
    det, _u, _v, _t = mt64(t, np.zeros((len(t), 3)), np.broadcast_to(d, (len(t), 3)), np.arange(len(t)))
    c[det < 0] = c[det < 0][:, ::-1]
    return _quads(c, ids)


TILE_ULP = 2.0 ** -33  # one ulp of 0.001f


def tilted_tiles(cornell_tris):
    """the Cornell box plus 12 tiles just above its floor whose normals have |n.x| within a few ulps of 0.001, the threshold
    that switches the tangent frame: y of the tiles near 6e-4, where one fp32 step of a vertex moves n.x by about an ulp"""
    corners, L, h = [], np.float32(0.35), np.float32(6e-4)
    for k, j in enumerate(range(-6, 6)):
        x0 = np.float32(-2.6 + 0.43 * k)
        dy = np.float32(0.001 * float(L) * (1 + j * 2.0 ** -21))
        corners.append([(x0, h, -0.3), (x0 + L, h - dy, -0.3), (x0 + L, h - dy, -0.3 - L), (x0, h, -0.3 - L)])
    tiles = _facing_quads(corners, np.full(12, 2), np.float64([0, -1, 0]))
    return np.concatenate([cornell_tris, tiles])


def _normal64(tris):
    p = [tris[k][:, :3].astype(np.float64) for k in ("p1", "p2", "p3")]
    n = np.cross(p[2] - p[0], p[1] - p[0])
    return n / np.linalg.norm(n, axis=1, keepdims=True)


# ---- comparisons -------------------------------------------------------------------------------------

CTR_FIELDS = ("rays_closest", "rays_any", "nodes", "tri_tests", "samples")


def assert_same_samples(got, want, msg):
    """bit-equal radiance; NaN only where the oracle has NaN, payloads masked (DESIGN.md section 2)"""
    gn, wn = np.isnan(got), np.isnan(want)
    np.testing.assert_array_equal(gn, wn, err_msg=f"{msg}: NaN positions")
    z = np.float32(0)
    np.testing.assert_array_equal(bits(np.where(gn, z, got)), bits(np.where(wn, z, want)), err_msg=f"{msg}: radiance")


def _oracle_tree_for(ob, sc, tris, mode, lbvh):
    if lbvh:
        return ob.make_bvh(*sc.bvh())
    bvh, keep, _b = oracle_tree(ob, tris, width=sc.mode_width(mode))
    return bvh, keep


W, H, NF = 96, 64, 3


def render_vs_oracle(dev, pt, ob, sc, tris, mats, mode, light, integrator, accel, lbvh=False, max_depth=8):
    """one ptb_render (LINEAR, collect_stats, frames_per_batch 2) against ora_render on the oracle's tree (or brute force)"""
    lkw = _light_kw(light, True) if light else {}
    prm = pt.default_params(width=W, height=H, n_frames=NF, mode=mode, accum=pt.ACCUM_LINEAR, max_depth=max_depth, ao_samples=4,
                            accel=accel, collect_stats=1, frames_per_batch=2, integrator=integrator, **lkw)
    fb, sb = dev.buffer(W * H * 16), dev.buffer(W * H * 32)
    try:
        ctr = dev.render(sc, prm, fb, sb, want_counters=True)
        rad, st = fb.read(np.float32).reshape(-1, 4), sb.read(pt.STATS_DTYPE)
    finally:
        fb.close(); sb.close()
    brute = accel == pt.ACCEL_BRUTE
    bvh, _keep = (None, None) if brute else _oracle_tree_for(ob, sc, tris, mode, lbvh)
    oprm = ob.default_params(W, H, n_frames=NF, mode=mode, accum=ob.ACCUM_LINEAR, max_depth=max_depth, ao_samples=4,
                             use_bvh=0 if brute else 1, **(_light_kw(light, False) if light else {}))
    want, wst, wctr = ob.render(oprm, tris, mats, bvh=bvh, want_stats=True)
    msg = f"mode {mode} integrator {integrator} accel {accel}"
    assert_same_samples(rad, want, msg)
    assert st.tobytes() == wst.tobytes(), f"{msg}: statistics"
    for f in CTR_FIELDS:
        assert ctr[f] == wctr[f], (msg, f, ctr[f], wctr[f])
    return want, wst


def shade_vs_oracle(dev, pt, ob, ora_shade, sc, tris, mats, mode, light, o, d, s, lbvh=False, max_depth=8):
    lkw = _light_kw(light, True) if light else {}
    prm = pt.default_params(mode=mode, max_depth=max_depth, ao_samples=8, **lkw)
    rad, st, ctr = _shade(dev, pt, sc, prm, o, d, s)
    bvh, _keep = _oracle_tree_for(ob, sc, tris, mode, lbvh)
    oprm = ob.default_params(1, 1, mode=mode, max_depth=max_depth, ao_samples=8, **(_light_kw(light, False) if light else {}))
    want, wst, wctr = ora_shade(oprm, tris, mats, o, d, s, bvh)
    msg = f"shade mode {mode}"
    assert_same_samples(rad, want, msg)
    assert st.tobytes() == wst.tobytes(), f"{msg}: statistics"
    for f in CTR_FIELDS:
        assert ctr[f] == wctr[f], (msg, f)
    return want, wst


# ---- part A without a device: what the tables and scenes claim to be --------------------------------

def test_scenes_reach_their_limits(pt, ob, cornell):
    tris, _ = cornell
    fl = flat_limit(tris)
    b = ob.build_bvh(fl)
    assert len(fl) == 64 and b["width"] == 1 and len(b["nodes"]) == 32
    assert (b["nodes"]["mask_hi"] != 0).any()  # the high half of the candidate mask is in use
    p = pt.build_bvh_host(fl, width=1)
    assert p["nodes"].tobytes() == b["nodes"].tobytes()
    tt = tilted_tiles(tris)
    nx = np.abs(_normal64(tt[36:])[:, 0])
    off = (nx - 0.001) / TILE_ULP
    assert (off < 0).sum() >= 3 and (off > 0).sum() >= 3 and (np.abs(off) <= 8).sum() >= 4, off


def test_garbage_in_unused_material_bytes_changes_nothing_in_the_oracle(ob, cornell):
    """albedo.w, emissive.w and the padding of every table hold NaN / 0xFF bytes; zeroing them leaves every mode's image,
    statistics and counters as they were"""
    tris, _ = cornell
    b = ob.build_bvh(tris)
    bvh, _keep = ob.make_bvh(b["nodes"], b["tri_order"])
    for name, m in tables(ob).items():
        clean = m.copy()
        raw = clean.view(np.uint8).reshape(18, 64)
        raw[:, 12:16] = 0
        raw[:, 28:32] = 0
        raw[:, 40:64] = 0
        for mode in (1, 3):
            prm = ob.default_params(48, 32, n_frames=2, mode=mode, accum=ob.ACCUM_REFERENCE, max_depth=6, ao_samples=4, use_bvh=1)
            a = ob.render(prm, tris, m, bvh=bvh, want_stats=True)
            c = ob.render(prm, tris, clean, bvh=bvh, want_stats=True)
            assert_same_samples(a[0], c[0], f"{name} mode {mode}")
            assert a[1].tobytes() == c[1].tobytes() and a[2] == c[2]


def test_the_matrix_reaches_its_cases(ob, cornell):
    """on the oracle: NaN samples occur, paths end on an unknown type, DIRECT has lit and unlit samples under each light"""
    tris, _ = cornell
    T = tables(ob)
    b = ob.build_bvh(tris)
    bvh, _keep = ob.make_bvh(b["nodes"], b["tri_order"])
    prm = lambda **kw: ob.default_params(W, H, n_frames=1, accum=ob.ACCUM_LINEAR, max_depth=8, use_bvh=1, **kw)
    fb, _st, _ = ob.render(prm(mode=3), tris, T["ggx"], bvh=bvh, want_stats=True)
    assert np.isnan(fb[:, :3]).any(axis=1).mean() > 0.01
    fb, _st, _ = ob.render(prm(mode=3), tris, T["albedo"], bvh=bvh, want_stats=True)
    assert np.isinf(fb[:, 0]).any() and np.isnan(fb[:, 0]).any()  # masks overflow, and inf x 0 emission makes NaN
    fb, st, _ = ob.render(prm(mode=3), tris, T["types"], bvh=bvh, want_stats=True)
    ended = np.isin(st["quad"], UNKNOWN_TYPE_QUADS) & (st["count"] == 1)
    assert ended.mean() > 0.3, ended.mean()
    bd = ob.build_bvh(tris, width=4)
    bvh4, _k4 = ob.make_bvh(bd["nodes"], bd["tri_order"])
    for name, light in lights(ob, tris).items():
        _fb, st, _ = ob.render(prm(mode=2, **_light_kw(light, False)), tris, T["albedo"], bvh=bvh4, want_stats=True)
        hit = st["tri"] >= 0
        if name == "degenerate":
            assert (st["count"][hit] == 0).all()
        else:
            assert (st["count"][hit] == 1).any() and (st["count"][hit] == 0).any(), name


# ---- part A on the B200 ------------------------------------------------------------------------------

def _forms(pt, tris):
    """name -> (triangles, scene kwargs, tuning knob 2 value, built by the LBVH)"""
    tess = pt.tessellate(tris, 12)
    return {
        "flat": (tris, {}, 0, False),
        "wide4": (tris, dict(bvh_params=pt.bvh_params(force_width=4)), 0, False),
        "tess": (tess, {}, 0, False),
        "tess-smem-stack": (tess, {}, 2, False),
        "tess-lbvh": (tess, dict(gpu_build=True), 0, True),
        "flat64": (flat_limit(tris), {}, 0, False),
        "tilted": (tilted_tiles(tris), {}, 0, False),
    }


FORM_WIDTH = {"flat": 1, "wide4": 4, "tess": 2, "tess-smem-stack": 2, "tess-lbvh": 2, "flat64": 1, "tilted": 1}


@pytest.mark.gpu
@pytest.mark.parametrize("form", list(FORM_WIDTH))
def test_render_equals_the_oracle_over_materials_and_lights(dev, pt, ob, cornell, form):
    """ptb_render, megakernel and wavefront (and brute force on the Cornell FLAT scene), every mode, DIRECT under every light,
    every material table: bit-equal to ora_render on the oracle's own tree"""
    tris0, _ = cornell
    tris, kw, stack, lbvh = _forms(pt, tris0)[form]
    accels = (pt.ACCEL_BVH, pt.ACCEL_BRUTE) if form == "flat" else (pt.ACCEL_BVH,)
    dev.set_tuning(2, stack)
    try:
        for name, mats in tables(ob).items():
            sc = dev.scene(tris, mats, **kw)
            try:
                assert sc.info()["width"] == FORM_WIDTH[form]
                if form == "flat64":
                    assert sc.info()["n_nodes"] == 32 and len(tris) == 64
                for mode, ln in _mode_variants(ob, tris0):
                    light = lights(ob, tris)[ln] if ln else None
                    for integ in (pt.INTEGRATOR_MEGAKERNEL, pt.INTEGRATOR_WAVEFRONT):
                        for accel in accels:
                            try:
                                render_vs_oracle(dev, pt, ob, sc, tris, mats, mode, light, integ, accel, lbvh=lbvh)
                            except AssertionError as e:
                                raise AssertionError(f"{form} {name} light {ln}: {e}") from None
            finally:
                sc.close()
    finally:
        dev.set_tuning(2, 0)


@pytest.mark.gpu
@pytest.mark.parametrize("form", list(FORM_WIDTH))
def test_shade_equals_the_oracle_over_materials_and_lights(dev, pt, ob, cornell, ora_shade, form):
    """ptb_scene_shade on rays no camera makes, every mode, DIRECT under every light, every material table"""
    tris0, _ = cornell
    tris, kw, stack, lbvh = _forms(pt, tris0)[form]
    o, d, s = _odd_rays(12_000, 300)
    if form == "tilted":  # straight down onto the tiles as well
        rng = np.random.default_rng(301)
        tgt = (tris["p1"][36:, :3] + tris["p3"][36:, :3]) / 2
        i = rng.integers(0, len(tgt), 4000)
        to = tgt[i] + rng.uniform(-0.15, 0.15, (4000, 3)) * [1, 0, 1] + [0, 2.0, 0]
        o = np.concatenate([o, to.astype(np.float32)])
        d = np.concatenate([d, np.tile(np.float32([0, -1, 0]), (4000, 1))])
        s = np.concatenate([s, rng.integers(0, 1 << 32, 4000, dtype=np.uint64).astype(np.uint32)])
    dev.set_tuning(2, stack)
    try:
        for name, mats in tables(ob).items():
            sc = dev.scene(tris, mats, **kw)
            try:
                for mode, ln in _mode_variants(ob, tris0):
                    light = lights(ob, tris)[ln] if ln else None
                    try:
                        shade_vs_oracle(dev, pt, ob, ora_shade, sc, tris, mats, mode, light, o, d, s, lbvh=lbvh)
                    except AssertionError as e:
                        raise AssertionError(f"{form} {name} light {ln}: {e}") from None
            finally:
                sc.close()
    finally:
        dev.set_tuning(2, 0)


@pytest.mark.gpu
def test_reference_accumulation_and_rgb8_of_nan_samples(dev, pt, ob, cornell):
    """the GGX table with roughness 0 makes NaN samples: the gamma-space running mean (ACCUM_REFERENCE) and the RGB8 output
    of the host entry point equal ora_render and ora_to_rgb8"""
    tris, _ = cornell
    mats = tables(ob)["ggx"]
    b = ob.build_bvh(tris)
    bvh, _keep = ob.make_bvh(b["nodes"], b["tri_order"])
    kw = dict(n_frames=3, mode=3, accum=ob.ACCUM_REFERENCE, max_depth=8)
    want, _, _ = ob.render(ob.default_params(W, H, use_bvh=1, **kw), tris, mats, bvh=bvh)
    assert np.isnan(want[:, :3]).any()
    for integ in (pt.INTEGRATOR_MEGAKERNEL, pt.INTEGRATOR_WAVEFRONT):
        got, _, _ = dev.render_host(tris, mats, pt.default_params(width=W, height=H, integrator=integ, **kw))
        assert_same_samples(got, want, f"reference accumulation, integrator {integ}")
        u8, _, _ = dev.render_host(tris, mats, pt.default_params(width=W, height=H, integrator=integ, output=pt.OUTPUT_RGB8, **kw))
        np.testing.assert_array_equal(u8, ob.to_rgb8(want))


# ---- part B: float64 references ----------------------------------------------------------------------

def _oracle_shader(ob, ora_shade):
    def run(tris, mats, o, d, s, **kw):
        bvh, _keep, _b = oracle_tree(ob, tris)
        prm = ob.default_params(1, 1, **kw)
        rad, st, _ = ora_shade(prm, tris, mats, o, d, s, bvh)
        return rad, st
    return run


def _device_shader(dev, pt):
    def run(tris, mats, o, d, s, **kw):
        sc = dev.scene(tris, mats)
        try:
            rad, st, _ = _shade(dev, pt, sc, pt.default_params(**kw), o, d, s)
        finally:
            sc.close()
        return rad, st
    return run


@pytest.fixture(params=["oracle", pytest.param("device", marks=pytest.mark.gpu)])
def shader(request, ob, ora_shade):
    if request.param == "oracle":
        return _oracle_shader(ob, ora_shade)
    return _device_shader(request.getfixturevalue("dev"), request.getfixturevalue("pt"))


def _mat(ob, n=1, albedo=(0.7, 0.7, 0.7), emissive=(0, 0, 0), roughness=0.0, typ=1):
    m = np.zeros(n, ob.MATERIAL_DTYPE)
    m["albedo"][:, :3], m["emissive"][:, :3], m["roughness"], m["type"] = albedo, emissive, roughness, typ
    m["albedo"][:, 3] = m["emissive"][:, 3] = 1.0
    return m


def furnace_cube():
    """the closed cube [-1, 1]^3, six quads facing inwards"""
    v = np.float32([[x, y, z] for x in (-1, 1) for y in (-1, 1) for z in (-1, 1)])
    faces = [(0, 1, 3, 2), (4, 6, 7, 5), (0, 4, 5, 1), (2, 3, 7, 6), (0, 2, 6, 4), (1, 5, 7, 3)]
    c = np.stack([v[list(f)] for f in faces])
    return _facing_quads(c, np.zeros(6, np.int32), c.mean(1))


FURNACE_A, FURNACE_E = 0.6, 0.05  # 3E = 0.15, not the background's 0.45
FURNACE_RTOL_PER_BOUNCE = 1e-7
FURNACE_MAX_ESCAPES = 0.025


@pytest.mark.parametrize("tess", [1, 14])
def test_furnace_samples_are_the_float64_geometric_sums(pt, ob, shader, tess):
    """a sample with count k is 3E sum_{j<k} a^j (last segment hit) or 3E sum_{j<k-1} a^j + a^(k-1) 0.45 (it escaped, through
    the 0.01 origin offset near an edge); FLAT cube and the tessellated one (binary tree, the C5 path kernel)"""
    cube = furnace_cube()
    tris = cube if tess == 1 else pt.tessellate(cube, tess)
    assert (len(tris) == 12) if tess == 1 else (ob.build_bvh(tris)["width"] == 2)
    mats = _mat(ob, albedo=(FURNACE_A,) * 3, emissive=(FURNACE_E,) * 3)
    rng = np.random.default_rng(400 + tess)
    n = 50_000
    o = rng.uniform(-0.9, 0.9, (n, 3)).astype(np.float32)
    d = rng.normal(size=(n, 3))
    d = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)
    s = rng.integers(0, 1 << 32, n, dtype=np.uint64).astype(np.uint32)
    a, e3 = np.float64(np.float32(FURNACE_A)), 3 * np.float64(np.float32(FURNACE_E))
    for depth in (1, 2, 5, 8):
        rad, st = shader(tris, mats, o, d, s, mode=3, max_depth=depth)
        k = st["count"].astype(np.int64)
        assert (k >= 1).all() and (k <= depth).all()
        geo = lambda m: (1 - a ** m) / (1 - a)
        hit = e3 * geo(k)
        esc = e3 * geo(k - 1) + a ** (k - 1) * 0.45
        r = rad[:, :3].astype(np.float64)
        err_hit = np.abs(r - hit[:, None]).max(1) / hit
        err_esc = np.abs(r - esc[:, None]).max(1) / esc
        err = np.minimum(err_hit, err_esc)
        escaped = err_esc < err_hit
        print(f"furnace tess {tess} depth {depth}: max rel err {err.max():.3g}, per bounce {(err / k).max():.3g}, "
              f"escapes {escaped.mean():.4f}")
        assert (err <= FURNACE_RTOL_PER_BOUNCE * k).all(), (depth, err.max())
        assert escaped.mean() <= FURNACE_MAX_ESCAPES
        assert (st["count"] == depth).mean() > 0.9


# DIRECT's expectation under one parallelogram light: floor y = 0 facing up, light at y = 1 facing down
LIGHT = ([-0.5, 1.0, -0.5], [1.2, 0.0, 0.0], [0.0, 0.0, 0.8])
LE = (2.0, 3.0, 4.0)
FLOOR_ALBEDO = (0.6, 0.5, 0.4)
POINTS = {"under": (0.1, 0.1), "side": (1.5, 0.3), "grazing": (12.0, 0.0)}
N_SEEDS = 1 << 20


def _floor_scene(ob, material, occluder):
    floor = _facing_quads([[(-30, 0, -30), (30, 0, -30), (30, 0, 30), (-30, 0, 30)]], [0], np.float64([0, -1, 0]))
    parts = [floor]
    if occluder == "far":  # a plane at y = 0.3 over z > 2: shadows points at z = 10, faces down (invisible from above)
        parts.append(_facing_quads([[(-30, 0.3, 2), (30, 0.3, 2), (30, 0.3, 30), (-30, 0.3, 30)]], [0], np.float64([0, 1, 0])))
    elif occluder == "near":  # a plate 0.1 below the light, wider than it
        parts.append(_facing_quads([[(-0.8, 0.9, -0.8), (1.0, 0.9, -0.8), (1.0, 0.9, 0.6), (-0.8, 0.9, 0.6)]], [0],
                                   np.float64([0, 1, 0])))
    mats = np.concatenate([material, _mat(ob, emissive=LE)])
    return np.concatenate(parts), mats


def _form_factor(x, verts):
    """Lambert's closed form: the form factor from a point with normal +y to a polygon, in float64"""
    R = [(v - x) / np.linalg.norm(v - x) for v in verts]
    f = 0.0
    for i in range(len(R)):
        a, b = R[i], R[(i + 1) % len(R)]
        c = np.cross(a, b)
        f += np.arccos(np.clip(np.dot(a, b), -1, 1)) * c[1] / np.linalg.norm(c)
    return abs(f) / (2 * np.pi)


def _ggx_expectation(x, rough, albedo):
    """float64 quadrature over the light of DIRECT's f * Le * 3 * cos_s * cos_l / r^2 (wo = +y, n = +y)"""
    from scipy import integrate

    p1, ea, eb = (np.float64(v) for v in LIGHT)
    area = np.linalg.norm(np.cross(ea, eb))
    r2 = rough * rough

    def g(b, a):
        L = p1 + a * ea + b * eb - x
        dist2 = L @ L
        wi = L / np.sqrt(dist2)
        cos_s = wi[1]
        cos_l = wi[1]  # the light's normal is -y
        h = wi + [0, 1, 0]
        ch = h[1] / np.linalg.norm(h)
        D = r2 / np.pi / (ch * ch * (r2 - 1) + 1) ** 2
        return D / (4 * cos_s) * 2 * cos_s * cos_l / dist2 * area

    val, _ = integrate.dblquad(g, 0, 1, 0, 1, epsabs=1e-12, epsrel=1e-10)
    return np.array(albedo) * np.array(LE) * 3 * val


@pytest.mark.parametrize("floor", ["diffuse", "ggx0.3", "ggx1.0"])
def test_direct_mean_equals_the_float64_expectation(ob, shader, floor):
    """2^20 seeds per point straight under the light, off to the side and near grazing to its plane: the mean equals
    albedo 3 Le F (Lambert's polygon form factor) on a diffuse floor, float64 quadrature of DIRECT's own integrand on a GGX
    floor, within 5 standard errors"""
    rough = 0.0 if floor == "diffuse" else float(floor[3:])
    material = _mat(ob, albedo=FLOOR_ALBEDO, roughness=rough, typ=1 if floor == "diffuse" else 2)
    tris, mats = _floor_scene(ob, material, "far")
    p1, ea, eb = (np.float64(v) for v in LIGHT)
    verts = [p1, p1 + ea, p1 + ea + eb, p1 + eb]
    for name, (px, pz) in POINTS.items():
        x = np.float64([px, 0, pz])
        o = np.tile(np.float32([px, 0.5, pz]), (N_SEEDS, 1))
        d = np.tile(np.float32([0, -1, 0]), (N_SEEDS, 1))
        s = np.arange(N_SEEDS, dtype=np.uint32) * np.uint32(2654435761)
        rad, st = shader(tris, mats, o, d, s, mode=2, light_quad=1, light_p1=LIGHT[0], light_ea=LIGHT[1], light_eb=LIGHT[2])
        assert (st["tri"] >= 0).all() and (st["count"] == 1).all()
        if floor == "diffuse":
            want = np.array(FLOOR_ALBEDO) * 3 * np.array(LE) * _form_factor(x, verts)
        else:
            want = _ggx_expectation(x, rough, FLOOR_ALBEDO)
        r = rad[:, :3].astype(np.float64)
        mean, se = r.mean(0), r.std(0) / np.sqrt(N_SEEDS)
        z = np.abs(mean - want) / se
        print(f"DIRECT {floor} {name}: mean {mean}, float64 {want}, {z.max():.2f} standard errors")
        assert (z <= 5).all(), (name, mean, want, z)


@pytest.mark.parametrize("occluder", ["far", "near"])
def test_direct_fully_shadowed_point_is_its_emission(ob, shader, occluder):
    """an occluder far from the light (a plane near the floor) and one 0.1 below it block every shadow ray: the sample is
    exactly the surface's own emission x 3"""
    material = _mat(ob, albedo=FLOOR_ALBEDO, emissive=(0.25, 0.5, 0.0))
    tris, mats = _floor_scene(ob, material, occluder)
    px, pz = (0.0, 10.0) if occluder == "far" else (0.1, -0.1)
    n = 1 << 16
    o = np.tile(np.float32([px, 0.5, pz]), (n, 1))
    d = np.tile(np.float32([0, -1, 0]), (n, 1))
    s = np.arange(n, dtype=np.uint32) * np.uint32(2246822519)
    rad, st = shader(tris, mats, o, d, s, mode=2, light_quad=1, light_p1=LIGHT[0], light_ea=LIGHT[1], light_eb=LIGHT[2])
    assert (st["tri"] >= 0).all() and (st["count"] == 0).all()
    want = np.float32(1.0) * np.float32([0.25, 0.5, 0.0]) * np.float32(3.0)
    np.testing.assert_array_equal(bits(rad[:, :3]), np.broadcast_to(bits(want), (n, 3)))


# ---- part B: per-sample DIRECT and AO against float64 -------------------------------------------------

def lcg_draws(seeds, n):
    """n draws of GenerateColors.cl:61-71 per seed, shape (n, len(seeds)): the integer steps are exact, so these are the very
    fp32 values both sides draw (returned as float64)"""
    s = np.array(seeds, np.uint32)
    out = np.empty((n, len(s)), np.float32)
    for k in range(n):
        s = (s ^ np.uint32(61)) ^ (s >> np.uint32(16))
        s = s + (s << np.uint32(3))
        s = s ^ (s >> np.uint32(4))
        s = s * np.uint32(0x27D4EB2D)
        s = s ^ (s >> np.uint32(15))
        s = np.uint32(1103515245) * s + np.uint32(12345)
        out[k] = s.astype(np.float32) * np.float32(2.3283064365386963e-10)
    return out.astype(np.float64)


def test_lcg_draws_are_the_oracles(ob):
    states, values = ob.rng_kat(17, 5, 6)
    s0 = np.uint32(17) + np.uint32(ob.lib().ora_hash_uint32(5))
    np.testing.assert_array_equal(lcg_draws([s0], 6)[:, 0], values.astype(np.float64))


MARGIN = 1e-5  # float64 decisions closer than this to their threshold (normalised det, barycentrics, t) are not clear


def segment_blocked64(tris, o, d, tmax, m=MARGIN, chunk=4096):
    """float64 any-hit over every triangle (one-sided, 0 < t < tmax) -> (blocked, clear): clear when some triangle clearly
    blocks the segment or every triangle clearly does not"""
    p = [tris[k][:, :3].astype(np.float64) for k in ("p1", "p2", "p3")]
    scale = np.linalg.norm(p[1] - p[0], axis=1) * np.linalg.norm(p[2] - p[0], axis=1)
    blocked, clear = np.zeros(len(o), bool), np.zeros(len(o), bool)
    with np.errstate(divide="ignore", invalid="ignore"):
        for s in range(0, len(o), chunk):
            det, u, v, t = mt64(tris, o[s:s + chunk], d[s:s + chunk])
            dn, mb, tm = det / scale, np.minimum(np.minimum(u, v), 1 - u - v), tmax[s:s + chunk, None]
            hit = (dn > m) & (mb > m) & (t > m) & (t < tm - m)
            miss = (dn < -m) | ((dn > m) & ((mb < -m) | (t < -m) | (t > tm + m)))
            blocked[s:s + chunk] = hit.any(1)
            clear[s:s + chunk] = hit.any(1) | (hit | miss).all(1)
    return blocked, clear


def _unit64(v):
    return v / np.linalg.norm(v, axis=-1, keepdims=True)


SOUP_LIGHT = ([-0.6, 2.0, -0.6], [1.2, 0.0, 0.0], [0.0, 0.0, 1.2])  # faces down
SOUP_LE = (2.0, 3.0, 4.0)
SOUP_MATERIALS = ((1, 0.0), (2, 0.3), (2, 1.0), (2, 0.05))  # (type, roughness) of materials 0-3; material 4 is the light


def occluder_soup(ob):
    """a 4 x 4 floor of four materials under 80 random occluder triangles of every orientation, and the light's material"""
    rng = np.random.default_rng(500)
    floor = _facing_quads([[(-2, 0, -2), (0, 0, -2), (0, 0, 0), (-2, 0, 0)], [(0, 0, -2), (2, 0, -2), (2, 0, 0), (0, 0, -2 + 2)],
                           [(-2, 0, 0), (0, 0, 0), (0, 0, 2), (-2, 0, 2)], [(0, 0, 0), (2, 0, 0), (2, 0, 2), (0, 0, 2)]],
                          np.arange(4), np.float64([0, -1, 0]))
    c = rng.uniform([-1.5, 0.2, -1.5], [1.5, 1.2, 1.5], (80, 3))
    occ = _triangles(*(c + rng.normal(size=(80, 3)) * 0.15 for _ in range(3)))
    occ["id"] = rng.integers(0, 4, 80)
    mats = np.concatenate([_mat(ob, albedo=(0.6, 0.5, 0.4), emissive=(0.1, 0.0, 0.05), roughness=r, typ=t) for t, r in SOUP_MATERIALS]
                          + [_mat(ob, emissive=SOUP_LE)])
    return np.concatenate([floor, occ]), mats


def soup_rays(tris, n, seed):
    """rays aimed at triangle interiors (barycentric margin >= 0.05) from the side each triangle faces, 0.3 to 3 away"""
    rng = np.random.default_rng(seed)
    b = rng.dirichlet([1, 1, 1], 4 * n)
    b = b[b.min(1) >= 0.05][:n]
    i = rng.integers(0, len(tris), n)
    p = [tris[k][i, :3].astype(np.float64) for k in ("p1", "p2", "p3")]
    tgt = b[:, :1] * p[0] + b[:, 1:2] * p[1] + b[:, 2:] * p[2]
    away = np.cross(p[2] - p[0], p[1] - p[0])  # rays along it hit the front face
    u = _unit64(rng.normal(size=(n, 3)))
    u = np.where((u * away).sum(1, keepdims=True) < 0, -u, u)
    o = (tgt - u * rng.uniform(0.3, 3.0, (n, 1))).astype(np.float32)
    d = _unit64(tgt - o.astype(np.float64)).astype(np.float32)
    return o, d, i, rng.integers(0, 1 << 32, n, dtype=np.uint64).astype(np.uint32)


def _primary64(tris, o, d, target):
    """float64 hit point and the normal facing the ray (GenerateColors.cl:128-130, :243) on the aimed-at triangle"""
    o64, d64 = o.astype(np.float64), d.astype(np.float64)
    _det, _u, _v, t = mt64(tris, o64, d64, target)
    p = [tris[k][target, :3].astype(np.float64) for k in ("p1", "p2", "p3")]
    n = _unit64(np.cross(p[2] - p[0], p[1] - p[0]))
    n = np.where((n * d64).sum(1, keepdims=True) < 0, n, -n)
    return o64 + t[:, None] * d64, n


def _ggx_d64(c, rough):
    r2 = rough * rough
    x = c * c * (r2 - 1) + 1
    return r2 / np.pi / (x * x), 2 * np.abs(c * c * (r2 - 1)) / x  # D and its condition number


DIRECT_C = 600  # rtol = DIRECT_C * 2^-24 * (1 + kappa); 296 measured on the oracle
DIRECT_MAX_EXCLUDED = 0.04  # 1.8 % measured
AO_MAX_EXCLUDED = 0.03  # 1.0 % measured
COS_MARGIN = 1e-2


def _aimed(ob, tris, o, d, target, st):
    """samples whose primary hit is the aimed-at triangle, clearly so in float64 and so in fp32"""
    win = clear_winner64(tris, o, d)
    return (win == target) & (st["tri"] == target)


def test_direct_per_sample_equals_float64(ob, shader):
    """DIRECT per sample on a floor of four materials under occluders: where every float64 decision has a clear margin,
    `count` is float64's shadow-ray visibility exactly and the radiance agrees to DIRECT_C 2^-24 (1 + kappa)"""
    tris, mats = occluder_soup(ob)
    o, d, target, s = soup_rays(tris, 40_000, 501)
    rad, st = shader(tris, mats, o, d, s, mode=2, light_quad=4, light_p1=SOUP_LIGHT[0], light_ea=SOUP_LIGHT[1],
                     light_eb=SOUP_LIGHT[2])
    aimed = _aimed(ob, tris, o, d, target, st)
    assert aimed.mean() > 0.6
    p, n = _primary64(tris, o, d, target)
    xi = lcg_draws(s, 2)
    lp, ea, eb = (np.float64(v) for v in SOUP_LIGHT)
    L = lp + xi[0][:, None] * ea + xi[1][:, None] * eb - p
    dist2 = (L * L).sum(1)
    dist = np.sqrt(dist2)
    wi = L / dist[:, None]
    lc = np.cross(ea, eb)
    area, nl = np.linalg.norm(lc), _unit64(lc)
    cos_s, cos_l = (wi * n).sum(1), -(wi @ nl)
    lit = (cos_s > 0) & (cos_l > 0)
    blocked, clear = segment_blocked64(tris, p + 0.01 * wi, wi, dist - 0.02)
    count = lit & ~blocked
    m = mats[tris["id"][target]]
    typ, rough = m["type"], m["roughness"].astype(np.float64)
    wo = -d.astype(np.float64)
    cos_h = (n * _unit64(wo + wi)).sum(1)
    D, kappa = _ggx_d64(cos_h, rough)
    spec = typ == 2
    albedo = m["albedo"][:, :3].astype(np.float64)
    f = np.where(spec[:, None], (D / (4 * cos_s * (wo * n).sum(1)))[:, None] * albedo * 2, albedo / np.pi)
    kappa = np.where(spec, kappa, 0.0)
    want = m["emissive"][:, :3].astype(np.float64) * 3
    want = want + np.where(count[:, None], f * (np.float64(SOUP_LE) * 3) * (cos_s * cos_l / dist2 * area)[:, None], 0.0)
    want = np.maximum(want, 0.0)
    cos_o = (wo * n).sum(1)  # a grazing primary ray magnifies the rounding of t into the hit point by 1 / cos_o
    keep = aimed & (np.minimum(np.minimum(np.abs(cos_s), np.abs(cos_l)), cos_o) > COS_MARGIN) & (clear | ~lit)
    excluded = 1 - keep.sum() / aimed.sum()
    np.testing.assert_array_equal(st["count"][keep], count[keep].astype(np.uint32))
    err = np.abs(rad[keep, :3] - want[keep]).max(1) / (np.abs(want[keep]).max(1) * 2.0 ** -24 * (1 + kappa[keep]))
    print(f"DIRECT per sample: {keep.sum()} kept, excluded {excluded:.4f}, lit {count[keep].mean():.3f}, "
          f"max err {err.max():.1f} x 2^-24 (1 + kappa), 99.9 % {np.quantile(err, 0.999):.1f}, GGX kappa up to {kappa[keep].max():.0f}")
    assert excluded <= DIRECT_MAX_EXCLUDED
    assert 0.2 < count[keep].mean() < 0.9 and (spec[keep] & count[keep]).any()
    assert err.max() <= DIRECT_C, err.max()


AO_MAX_DIST, AO_NS = 1.0, 8


def test_ao_per_sample_equals_float64(ob, shader):
    """AO per sample: where every AO ray's float64 decision and the tangent-frame choice (|n.x| against 0.001) have a clear
    margin, the open count equals float64's (origin p + 0.01 wi, tmax = ao_max_dist)"""
    tris, mats = occluder_soup(ob)
    o, d, target, s = soup_rays(tris, 20_000, 502)
    rad, st = shader(tris, mats, o, d, s, mode=1, ao_samples=AO_NS, ao_max_dist=AO_MAX_DIST)
    aimed = _aimed(ob, tris, o, d, target, st)
    p, n = _primary64(tris, o, d, target)
    axis = np.where((np.abs(n[:, 0]) > 0.001)[:, None], [0.0, 1.0, 0.0], [1.0, 0.0, 0.0])
    t = _unit64(np.cross(axis, n))
    b = np.cross(n, t)
    xi = lcg_draws(s, 2 * AO_NS)
    open_, clear = np.zeros(len(o), np.uint32), np.abs(np.abs(n[:, 0]) - 0.001) > 1e-6
    for k in range(AO_NS):
        phi, s2 = 2 * np.pi * xi[2 * k], xi[2 * k + 1]
        wi = _unit64(b * (np.cos(phi) * np.sqrt(s2))[:, None] + t * (np.sin(phi) * np.sqrt(s2))[:, None]
                     + n * np.sqrt(1 - s2)[:, None])
        blk, clr = segment_blocked64(tris, p + 0.01 * wi, wi, np.full(len(o), AO_MAX_DIST))
        open_ += ~blk
        clear &= clr
    keep = aimed & clear
    excluded = 1 - keep.sum() / aimed.sum()
    print(f"AO per sample: {keep.sum()} kept, excluded {excluded:.4f}, mean open {open_[keep].mean() / AO_NS:.3f}, "
          f"frames (1,0,0) {(np.abs(n[keep, 0]) <= 0.001).mean():.3f}")
    np.testing.assert_array_equal(st["count"][keep], open_[keep])
    np.testing.assert_array_equal(bits(rad[keep, 0]), bits(np.float32(open_[keep]) / np.float32(AO_NS)))
    assert excluded <= AO_MAX_EXCLUDED
    assert 0.2 < open_[keep].mean() / AO_NS < 0.9 and (np.abs(n[keep, 0]) <= 0.001).any() and (np.abs(n[keep, 0]) > 0.001).any()
