"""ptb_bvh_params.builder = PTB_BUILDER_SAH: the host's binned-SAH tree built on the device (csrc/sah_build.cuh).

The reference for every check is ptb_scene_create(force_width = 2) on the same records: the same ptb_scene_info, node bytes,
tri_order, quantised nodes and grid, through both device entry points (ptb_scene_create_gpu and ptb_scene_create_from_device),
on generated scenes, the Cornell box and its tessellations, scenes that keep the device's level-by-level phase busy for many
levels, every combination of the SAH parameters, and the 2M-triangle C5 scene.  The trees also equal the oracle's own builder.
Renders in every mode (megakernel and wavefront), intersect and shade results on a device-built SAH scene equal those on the
host-built one bit for bit.
"""
import ctypes as C
import os
import re

import numpy as np
import pytest

from conftest import ROOT, assert_same_tree, bits, oracle_tree
from test_traversal_scenes import SCENES, duplicated, same_centroid, scene as generated_scene, soup

# ---- no device needed --------------------------------------------------------------------------------


def test_bvh_params_layout(pt):
    assert C.sizeof(pt.BvhParams) == 32
    assert pt.BvhParams.builder.offset == 24 and pt.BvhParams.reserved.offset == 28


def test_header_builder_values_match_the_binding(pt):
    with open(os.path.join(ROOT, "include", "ptb200.h")) as f:
        h = f.read()
    got = {m.group(1): int(m.group(2)) for m in re.finditer(r"#define PTB_BUILDER_(\w+) (\d+)", h)}
    assert got == {"LBVH": pt.BUILDER_LBVH, "SAH": pt.BUILDER_SAH} == {"LBVH": 0, "SAH": 1}
    assert pt.bvh_params().builder == pt.BUILDER_LBVH  # the default keeps today's device tree


def test_host_builders_ignore_the_field(pt):
    tris = soup(300, 5)
    a = pt.build_bvh_host(tris, pt.bvh_params(), width=2)
    b = pt.build_bvh_host(tris, pt.bvh_params(builder=pt.BUILDER_SAH), width=2)
    c = pt.build_bvh_host(tris, pt.bvh_params(builder=7), width=2)
    for x in (b, c):
        assert x["nodes"].tobytes() == a["nodes"].tobytes() and np.array_equal(x["tri_order"], a["tri_order"])


# ---- helpers -----------------------------------------------------------------------------------------

def _upload(dev, arr):
    b = dev.buffer(arr.nbytes)
    b.write(arr)
    return b


def _from_device(dev, tris, mats, bp):
    tb, mb = _upload(dev, tris), _upload(dev, mats)
    try:
        return dev.scene_from_device(tb, mb, bp)
    finally:
        tb.close(); mb.close()


def _sah(pt, **kw):
    return pt.bvh_params(builder=pt.BUILDER_SAH, **kw)


def _host(pt, **kw):
    return pt.bvh_params(force_width=2, **kw)


def _tree(sc, quantized=True):
    """everything a binary scene is made of, as bytes"""
    nodes, order = sc.bvh()
    out = {"info": sc.info(), "nodes": nodes.tobytes(), "order": order.tobytes()}
    if quantized:
        q, lo, step = sc.bvh_quantized()
        out["q"] = q.tobytes()
        out["grid"] = bits(np.float32(lo + step)).tobytes()
    return out, nodes, order


def assert_same_scene(a, b, quantized=True):
    ta, _, _ = _tree(a, quantized)
    tb, _, _ = _tree(b, quantized)
    assert ta["info"] == tb["info"] and ta["info"]["width"] == 2
    for k in ta:
        assert ta[k] == tb[k], k


def _check_scene(dev, pt, ob, tris, mats, oracle=True, **kw):
    """both device entry points with the SAH builder == the host build == the oracle's builder"""
    ref = dev.scene(tris, mats, _host(pt, **kw))
    try:
        for sc in (dev.scene(tris, mats, _sah(pt, **kw), gpu_build=True), _from_device(dev, tris, mats, _sah(pt, **kw))):
            try:
                assert_same_scene(ref, sc)
            finally:
                sc.close()
        if oracle:
            nodes, order = ref.bvh()
            _bvh, _keep, b = oracle_tree(ob, tris, width=2, **kw)
            assert_same_tree(nodes, order, b)
            assert ref.info()["depth"] == b["depth"] and ref.info()["smem_nodes"] == b["bfs_nodes"]
    finally:
        ref.close()


def _with_ids(tris, n_mats):
    t = tris.copy()
    t["id"] = (np.arange(len(t)) // 2) % n_mats
    return t


# ---- on the B200 -------------------------------------------------------------------------------------

CASES = sorted(SCENES) + ["cornell", "tess2", "tess6", "tess20"]


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES)
def test_equals_the_host_tree(dev, pt, ob, cornell, case):
    tris, mats = cornell
    if case.startswith("tess"):
        tris = pt.tessellate(tris, int(case[4:]))
    elif case != "cornell":
        tris = generated_scene(case)
    _check_scene(dev, pt, ob, tris, mats)


LARGE = {
    "soup-200k": lambda: soup(200_000, 77, size=0.004),
    "centroid-20k": lambda: same_centroid(20_000, 78),    # every range takes the median fallback, large ranges too
    "dup-20k": lambda: duplicated(20_000, 79),
    "centroid-soup-mix": lambda: np.concatenate([same_centroid(6000, 80), soup(6000, 81)]),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(LARGE))
def test_large_ranges_equal_the_host_tree(dev, pt, ob, cornell, name):
    _check_scene(dev, pt, ob, LARGE[name](), cornell[1])


@pytest.mark.gpu
def test_every_parameter_combination_equals_the_host_tree(dev, pt, cornell):
    """max_leaf x n_bins x traverse_cost x smem_nodes on a scene with large ranges; smem_nodes 2, 3, 5, 1000 end the
    breadth-first prefix partway through a level"""
    tris = np.concatenate([soup(2500, 90), same_centroid(300, 91)])
    mats = cornell[1]
    combos = 0
    for max_leaf in (1, 2, 4, 8):
        for n_bins in (2, 3, 16, 256):
            for traverse_cost in (0.3, 1.2, 5.0):
                for smem_nodes in (1, 2, 3, 5, 1000, 1024, 1 << 20):
                    kw = dict(max_leaf=max_leaf, n_bins=n_bins, traverse_cost=traverse_cost, smem_nodes=smem_nodes)
                    ref = dev.scene(tris, mats, _host(pt, **kw))
                    sc = dev.scene(tris, mats, _sah(pt, **kw), gpu_build=True)
                    try:
                        assert_same_scene(ref, sc, quantized=smem_nodes == 1024), kw
                    finally:
                        ref.close(); sc.close()
                    combos += 1
    assert combos == 336


@pytest.mark.gpu
def test_c5_equals_the_host_tree_and_frame(dev, pt, cornell):
    """the 2,005,056-triangle C5 scene from a device buffer: the host tree byte for byte, one 4K PATH frame bit for bit, and
    two device builds give the same bytes"""
    tris, mats = cornell
    big = pt.tessellate(tris, 236)
    assert len(big) == 2_005_056
    host = dev.scene(big, mats)
    assert host.info()["width"] == 2
    a = _from_device(dev, big, mats, _sah(pt))
    b = _from_device(dev, big, mats, _sah(pt))
    ta = _tree(a)[0]
    assert ta == _tree(host)[0]
    assert ta == _tree(b)[0]
    b.close()
    prm = pt.default_params(width=3840, height=2160, n_frames=1, mode=pt.MODE_PATH, accum=pt.ACCUM_LINEAR, max_depth=8,
                            collect_stats=1)
    got = []
    for sc in (host, a):
        fb, sb = dev.buffer(3840 * 2160 * 16), dev.buffer(3840 * 2160 * 32)
        ctr = dev.render(sc, prm, fb, sb, want_counters=True)
        got.append((fb.read(np.uint32).tobytes(), sb.read(np.uint8).tobytes(), ctr))
        fb.close(); sb.close()
    assert got[0] == got[1]
    assert got[0][2]["rays_closest"] > 3840 * 2160
    a.close(); host.close()


@pytest.mark.gpu
@pytest.mark.parametrize("k", [6, 20])
def test_every_consumer_equals_the_host_scene(dev, pt, cornell, k):
    """renders of every mode (megakernel and wavefront; DIRECT takes its light from the scene's light table, light_ea = 0),
    intersect (closest and any) and shade: bit for bit, statistics and counters included"""
    from test_scene_from_device import assert_same_outputs

    tris, mats = cornell
    tris = pt.tessellate(tris, k)
    kw = dict(max_leaf=2, smem_nodes=300) if k == 20 else {}
    host = dev.scene(tris, mats, _host(pt, **kw))
    sc = _from_device(dev, tris, mats, _sah(pt, **kw))
    try:
        assert_same_scene(host, sc)
        assert_same_outputs(dev, pt, host, sc, tris)
    finally:
        host.close(); sc.close()


def _message(e):
    return str(e).split(": ", 2)[2]  # "ptb error -1: <entry point>: <verdict>"


@pytest.mark.gpu
def test_builder_values_are_checked(dev, pt, cornell):
    tris, mats = cornell
    tris = pt.tessellate(tris, 2)
    for builder in (2, -1, 100):
        with pytest.raises(pt.PtbError) as e:
            dev.scene(tris, mats, pt.bvh_params(builder=builder), gpu_build=True)
        assert "ptb_scene_create_gpu" in str(e.value) and f"builder = {builder}" in str(e.value)
        with pytest.raises(pt.PtbError) as e:
            _from_device(dev, tris, mats, pt.bvh_params(builder=builder))
        assert "ptb_scene_create_from_device" in str(e.value) and f"builder = {builder}" in str(e.value)
    # builder 0 is today's LBVH scene
    for gpu in (True, False):
        mk = (lambda bp: dev.scene(tris, mats, bp, gpu_build=True)) if gpu else (lambda bp: _from_device(dev, tris, mats, bp))
        a, b = mk(None), mk(pt.bvh_params(builder=pt.BUILDER_LBVH))
        assert a.info()["n_nodes"] == len(tris) - 1 and a.info()["smem_nodes"] == 1
        assert_same_scene(a, b)
        a.close(); b.close()


@pytest.mark.gpu
def test_existing_checks_hold_under_the_sah_builder(dev, pt, cornell):
    tris, mats = cornell
    tris = pt.tessellate(tris, 2)
    n = len(tris)

    def refused(bad, bp, both=True):
        msgs = []
        for gpu in ((True, False) if both else (False,)):
            with pytest.raises(pt.PtbError) as e:
                if gpu:
                    dev.scene(bad, mats, bp, gpu_build=True)
                else:
                    _from_device(dev, bad, mats, bp)
            msgs.append(_message(e.value))
        return msgs

    for i in (0, n // 2, n - 1):
        bad = tris.copy()
        bad["id"][i] = len(mats)
        assert refused(bad, _sah(pt)) == [f"triangle {i} has id {len(mats)} outside [0,{len(mats)})"] * 2
        for v in (np.nan, np.inf, -3.1e38):
            bad = tris.copy()
            bad["p2"][i, 1] = v
            assert refused(bad, _sah(pt)) == [f"triangle {i} has a non-finite vertex"] * 2
    for fw in (1, 4):
        (m,) = refused(tris, _sah(pt, force_width=fw), both=False)
        assert m.startswith(f"force_width = {fw}; only the binary form")
    for pad in (0.0, -1e-4, float("nan"), float("inf")):
        for m in refused(tris, _sah(pt, pad_rel=pad)):
            assert m.startswith("pad_rel must be a finite number > 0")
    # the refusals and repeated builds leave device memory where it was
    big = pt.tessellate(cornell[0], 40)
    free0 = None
    for it in range(12):
        s = _from_device(dev, big, mats, _sah(pt)) if it % 2 else dev.scene(big, mats, _sah(pt), gpu_build=True)
        s.close()
        if it == 1:
            free0 = dev.memory()[0]
    assert dev.memory()[0] >= free0 - (8 << 20)


@pytest.mark.gpu
def test_torch_tensors(pt, cornell):
    """records in CUDA tensors on torch's stream (Device.scene_from_device) with the SAH builder"""
    torch = pytest.importorskip("torch")
    tris, mats = cornell
    tess = _with_ids(soup(5000, 92), len(mats))
    src = torch.from_numpy(np.ascontiguousarray(tess).view(np.float32).reshape(-1, 16)).cuda()
    torch.cuda.synchronize()
    dev = pt.Device(0, stream=torch.cuda.current_stream().cuda_stream)
    try:
        ref = dev.scene(tess, mats, _host(pt))
        sc = dev.scene_from_device(src, mats, _sah(pt))
        assert_same_scene(ref, sc)
        sc.close(); ref.close()
    finally:
        dev.close()
