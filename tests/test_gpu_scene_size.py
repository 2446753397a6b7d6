"""Scenes beyond the 16-entry parameter block (device-memory scene tables) against the oracle, bit for bit."""
import os

import numpy as np
import pytest

from rayn_b200 import _lib as L
from rayn_b200 import configs
from rayn_b200.film import FrameInputs, Renderer
from rayn_b200.scene import BoxFold, MandelBox, SphereFold, SphereLight, Srgb, TracedSDF, Vec3

from helpers import CH, assert_bit_equal, random_rays

pytestmark = pytest.mark.gpu
TR = configs.frame_time_range(1)


def _inputs(res, samples, mb):
    integ = configs.PathTracingIntegrator(mb, 2)
    return FrameInputs(res[0], res[1], samples, integ), integ


def _render(world, cam, res, samples, mb, flags=0, max_paths=0, **kw):
    inp, integ = _inputs(res, samples, mb)
    r = Renderer(0, max_paths_per_pass=max_paths, flags=flags)
    try:
        r.upload_scene(world, cam)
        return r.render_host(inp, (16, 16), integ, TR, **kw)
    finally:
        r.close()


def _against_oracle(oracle, world, cam, res, samples, mb, what, flags=0):
    g = _render(world, cam, res, samples, mb, flags)
    inp, integ = _inputs(res, samples, mb)
    o, _ = oracle.render(world, cam, inp, (16, 16), integ, TR)
    for ch in CH:
        assert_bit_equal(g[ch], o[ch], f"{what} {ch}")
    assert float(o["color"].sum() + o["background"].sum()) > 0
    return g


def _with_lights(n_lights):
    """13 hitables, 6 materials and exactly n_lights lights (the extra lights have no emissive sphere)."""
    cam, w = configs.sphere_field((48, 32), 12, 2, 6, seed=5)
    rng = np.random.default_rng(9)
    while len(w.lights) < n_lights:
        p = rng.uniform(-2.0, 2.0, 3).astype(np.float32)
        w.lights.append(SphereLight(Vec3(*p), 0.1, Srgb(1.0, 0.8, 0.6) * 20.0))
    return cam, w


BOUNDARIES = {
    "hitables16": lambda: configs.sphere_field((48, 32), 15, 2, 6, seed=1),
    "hitables17": lambda: configs.sphere_field((48, 32), 16, 2, 6, seed=1),
    "materials16": lambda: configs.sphere_field((48, 32), 12, 2, 16, seed=2),
    "materials17": lambda: configs.sphere_field((48, 32), 12, 2, 17, seed=2),
    "lights16": lambda: _with_lights(16),
    "lights17": lambda: _with_lights(17),
    "max": lambda: configs.sphere_field((48, 32), 1023, 256, 1024, seed=3),
}


@pytest.mark.parametrize("case", sorted(BOUNDARIES))
def test_boundary_counts_bit_exact(oracle, case):
    cam, w = BOUNDARIES[case]()
    desc, _ = w.flatten(cam)
    if case == "max":
        assert (desc.n_hitables, desc.n_materials, desc.n_lights) == (L.RAYN_MAX_HITABLES, L.RAYN_MAX_MATERIALS, L.RAYN_MAX_LIGHTS)
    _against_oracle(oracle, w, cam, (48, 32), 1, 2, case)


def _field(**kw):
    return configs.sphere_field((64, 48), 499, 64, 300, seed=11, volume=True, **kw)


@pytest.mark.parametrize("variant", ["fold_all", "no_fold_all", "fractal_first", "fractal_middle", "fractal_last", "moving"])
def test_sphere_field_bit_exact(oracle, variant):
    kw = {"fold_all": {}, "no_fold_all": {}, "fractal_first": {"fractal_index": 0}, "fractal_middle": {"fractal_index": 250},
          "fractal_last": {"fractal_index": 500}, "moving": {"moving": True}}[variant]
    cam, w = _field(**kw)
    _against_oracle(oracle, w, cam, (64, 48), 2, 3, variant, flags=L.FLAG_NO_FOLD_ALL if variant == "no_fold_all" else 0)


def test_packet_order_identical_for_a_sphere_field(oracle):
    cam, w = configs.sphere_field((40, 24), 200, 8, 40, seed=4)
    inp, integ = _inputs((40, 24), 2, 2)
    r = Renderer(0)
    try:
        r.upload_scene(w, cam)
        r.enable_queue_log(True)
        r.render_host(inp, (16, 16), integ, TR)
        glog = r.read_queue_log()
    finally:
        r.close()
    _, info = oracle.render(w, cam, inp, (16, 16), integ, TR, n_threads=1, queue_log=True)

    def parse(log):
        out, i = {}, 0
        while i < len(log):
            depth, tile, ns = log[i:i + 3]
            out[(int(depth), int(tile))] = log[i + 3:i + 3 + ns].copy()
            i += 3 + ns
        return out
    g = {k: v for k, v in parse(glog).items() if len(v)}
    o = {k: v for k, v in parse(info["queue_log"]).items() if len(v)}
    assert set(g) == set(o)
    for k in o:
        assert np.array_equal(g[k], o[k]), f"shading queue differs at depth/tile {k}"
    assert any((v < 0).any() for v in o.values()), "no padded packet"


def test_stage_kernels_on_a_1000_sphere_scene(renderer, oracle):
    cam, w = configs.sphere_field((64, 64), 999, 16, 50, seed=6)
    desc, keep = w.flatten(cam)
    assert desc.n_hitables == 1000
    renderer.upload_scene_desc(desc)
    geo = {}
    for i in range(desc.n_hitables):
        h = desc.hitables[i]
        if h.kind == L.HITABLE_SPHERE:
            geo.setdefault(bytes(h)[8:24], []).append(i)
    dups = [v for v in geo.values() if len(v) > 1]
    assert dups
    o, d = random_rays(20_000, seed=21, spread=1.5)
    # rays straight at the duplicated spheres, so that the first-index-wins rule decides their hit object
    rng = np.random.default_rng(5)
    aim = []
    for v in dups:
        c = np.array(desc.hitables[v[0]].center, np.float32)
        for _ in range(200):
            src = rng.uniform(-3.0, 3.0, 3).astype(np.float32) + np.float32([0.0, 3.0, 0.0])
            aim.append((src, c + rng.uniform(-0.02, 0.02, 3).astype(np.float32)))
    ao = np.array([a for a, _ in aim], np.float32)
    ad = np.array([b - a for a, b in aim], np.float32)
    ad /= np.linalg.norm(ad, axis=1, keepdims=True)
    o, d = np.concatenate([o, ao]), np.concatenate([d, ad])
    for depth in (0, 2):
        gt, gobj = renderer.kat_closest_hit(depth, o, d)
        rt, robj = oracle.kat_closest_hit(desc, depth, o, d)
        assert (gobj == robj).all(), depth
        assert_bit_equal(gt, rt, f"closest-hit t depth {depth}")
    assert any(v[0] in set(robj.tolist()) for v in dups), "no ray ended on a duplicated sphere"
    assert not any(i in set(robj.tolist()) for v in dups for i in v[1:]), "a later duplicate won a tie"
    assert len(np.unique(robj)) >= 50
    s = rng.uniform(-3.0, 3.0, size=(20_000, 3)).astype(np.float32)
    e = rng.uniform(-3.0, 3.0, size=(20_000, 3)).astype(np.float32)
    g = renderer.kat_occluded(s, e)
    assert (g >= 0).all(), "early-out occlusion disagrees with the reference product form"
    assert_bit_equal(g, oracle.kat_occluded(desc, s, e), "occluded")
    assert 0.02 < g.mean() < 0.98


def test_golden_fixtures_through_the_scene_tables():
    from test_cpu_oracle import GOLD, GOLD_SUFFIX, GOLDEN_CASES
    r = Renderer(0, flags=L.FLAG_SCENE_TABLES)
    try:
        for name, (n, res, samples, mb) in sorted(GOLDEN_CASES.items()):
            c = configs.baseline_config(n, res=res, samples=samples, max_bounces=mb)
            inp = FrameInputs(res[0], res[1], c["samples"], c["integrator"])
            r.upload_scene(c["world"], c["camera"])
            g = r.render_host(inp, (16, 16), c["integrator"], TR)
            gold = np.load(os.path.join(GOLD, name + GOLD_SUFFIX + ".npz"))
            for ch in CH:
                assert_bit_equal(g[ch], gold[ch], f"golden {name} {ch} (scene tables)")
    finally:
        r.close()


def test_graph_replay_follows_the_uploaded_tables(oracle):
    res, samples, mb = (48, 32), 1, 2
    inp, integ = _inputs(res, samples, mb)
    cam_a, a = configs.sphere_field(res, 40, 4, 10, seed=1)
    cam_b, b = configs.sphere_field(res, 40, 4, 10, seed=2)
    small = configs.baseline_config(3, res=res, samples=samples, max_bounces=mb)
    want = {k: oracle.render(w, cam, inp, (16, 16), integ, TR)[0] for k, (cam, w) in
            {"a": (cam_a, a), "b": (cam_b, b), "small": (small["camera"], small["world"])}.items()}
    r = Renderer(0)
    try:
        for k, cam, w in [("a", cam_a, a), ("b", cam_b, b), ("b", cam_b, b), ("small", small["camera"], small["world"]), ("a", cam_a, a)]:
            r.upload_scene(w, cam)
            for rep in range(2):  # the second render of an upload replays the captured graph
                g = r.render_host(inp, (16, 16), integ, TR)
                assert r.stats().reserved_ == 1, "small frame did not run as a graph"
                for ch in CH:
                    assert_bit_equal(g[ch], want[k][ch], f"scene {k} render {rep} {ch}")
    finally:
        r.close()


def test_pass_size_and_sharding_do_not_change_a_large_scene_film(oracle):
    cam, w = configs.sphere_field((160, 96), 100, 8, 20, seed=8)
    full = _render(w, cam, (160, 96), 2, 2)
    inp, integ = _inputs((160, 96), 2, 2)
    r = Renderer(0, max_paths_per_pass=16 * 16 * 8 * 3)
    try:
        r.upload_scene(w, cam)
        f = r.render_host(inp, (16, 16), integ, TR)
        assert r.stats().passes > 1
    finally:
        r.close()
    for ch in CH:
        assert_bit_equal(f[ch], full[ch], f"pass-size {ch}")
    from rayn_b200.dist import shard_tiles
    from rayn_b200.film import tile_grid
    ntx, nty = tile_grid(160, 96, 16, 16)
    acc = {ch: np.zeros_like(full[ch]) for ch in CH}
    for rank in range(2):
        part = _render(w, cam, (160, 96), 2, 2, tile_list=shard_tiles(ntx, nty, rank, 2, "index"))
        for ch in CH:
            acc[ch] += part[ch]
    for ch in CH:
        assert_bit_equal(acc[ch], full[ch], f"sharded {ch}")
    o, _ = oracle.render(w, cam, inp, (16, 16), integ, TR, subsample_k=5)
    mask = o["alpha"] + o["background"].reshape(-1, 3).sum(1) + o["color"].reshape(-1, 3).sum(1) != 0
    assert mask.sum() > 0
    assert_bit_equal(full["color"].reshape(-1, 3)[mask], o["color"].reshape(-1, 3)[mask], "subset color")


def _over_sdf_limit():
    cam, w = configs.sphere_field((32, 32), 10, 2, 5)
    for _ in range(L.RAYN_MAX_SDF_HITABLES):
        w.hitables.push(TracedSDF(MandelBox(4, BoxFold(1.0), SphereFold(0.01, 1.9), -2.1), 1))
    return cam, w


@pytest.mark.parametrize("case,name", [
    ("hitables", "RAYN_MAX_HITABLES"), ("materials", "RAYN_MAX_MATERIALS"), ("lights", "RAYN_MAX_LIGHTS"), ("sdf", "RAYN_MAX_SDF_HITABLES")])
def test_limits_are_rejected_by_name_and_the_context_stays_usable(oracle, case, name):
    cam, w = {"hitables": lambda: configs.sphere_field((32, 32), 1024, 2, 5),
              "materials": lambda: configs.sphere_field((32, 32), 20, 2, 1025),
              "lights": lambda: configs.sphere_field((32, 32), 300, 257, 5),
              "sdf": _over_sdf_limit}[case]()
    desc, keep = w.flatten(cam)
    assert desc.n_hitables == 1025 or desc.n_materials == 1025 or desc.n_lights == 257 or case == "sdf"
    r = Renderer(0)
    try:
        with pytest.raises(L.RaynError) as e:
            r.upload_scene_desc(desc)
        assert e.value.code == L.RAYN_ERR_INVALID_ARG and name in str(e.value)
        cam2, ok = configs.sphere_field((32, 32), 40, 4, 10, seed=7)
        inp, integ = _inputs((32, 32), 1, 1)
        r.upload_scene(ok, cam2)
        g = r.render_host(inp, (16, 16), integ, TR)
        o, _ = oracle.render(ok, cam2, inp, (16, 16), integ, TR)
        for ch in CH:
            assert_bit_equal(g[ch], o[ch], f"after rejecting {case}: {ch}")
    finally:
        r.close()


@pytest.mark.skipif(L.MULADD_FUSED or L.LEGACY, reason="already inside a variant run")
def test_fused_mul_add_variant_passes_the_scene_size_suite():
    """The same file with the fused `mul_add` build of the kernels and the oracle (oracle/README.md A6)."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "pytest", "-x", "-q", "-m", "gpu", "-p", "no:cacheprovider", "tests/test_gpu_scene_size.py"], cwd=root,
                       env=dict(os.environ, RAYN_MULADD_FUSED="1"), capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-1500:]
    assert " passed" in r.stdout
