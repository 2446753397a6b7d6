"""Scenes beyond the parameter-block size: the public limits, the seeded `sphere_field` scene and the oracle at 1024 hitables
(no GPU needed)."""
import os
import re

import numpy as np

from rayn_b200 import _lib as L
from rayn_b200 import configs
from rayn_b200.film import FrameInputs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TR = configs.frame_time_range(1)


def test_limit_macros_match_the_python_binding():
    hdr = open(os.path.join(ROOT, "include", "rayn_b200.h")).read()
    macros = dict(re.findall(r"#define (RAYN_MAX_\w+) (\d+)", hdr))
    assert set(macros) == {"RAYN_MAX_HITABLES", "RAYN_MAX_MATERIALS", "RAYN_MAX_LIGHTS", "RAYN_MAX_SDF_HITABLES"}
    for name, value in macros.items():
        assert getattr(L, name) == int(value), name
    assert (L.RAYN_MAX_HITABLES, L.RAYN_MAX_MATERIALS, L.RAYN_MAX_LIGHTS, L.RAYN_MAX_SDF_HITABLES) == (1024, 1024, 256, 16)
    flag = int(re.search(r"#define RAYN_FLAG_SCENE_TABLES (\d+)", hdr).group(1))
    assert flag == L.FLAG_SCENE_TABLES
    others = [int(v) for v in re.findall(r"#define RAYN_FLAG_\w+ (\d+)", hdr)]
    assert others.count(flag) == 1, "RAYN_FLAG_SCENE_TABLES shares a bit with another flag"


def _flat(world, cam):
    desc, keep = world.flatten(cam)
    hit = [bytes(desc.hitables[i]) for i in range(desc.n_hitables)]
    mat = [bytes(desc.materials[i]) for i in range(desc.n_materials)]
    lig = [bytes(desc.lights[i]) for i in range(desc.n_lights)]
    return desc, hit, mat, lig


def test_sphere_field_is_seeded_and_has_the_requested_counts():
    cam, w = configs.sphere_field((64, 48), 500, 64, 300, seed=3)
    desc, hit, mat, lig = _flat(w, cam)
    assert (desc.n_hitables, desc.n_materials, desc.n_lights) == (501, 300, 64)
    kinds = [desc.hitables[i].kind for i in range(desc.n_hitables)]
    assert kinds.count(L.HITABLE_MANDELBOX) == 1 and kinds[1] == L.HITABLE_MANDELBOX
    assert desc.hitables[0].kind == L.HITABLE_SPHERE and desc.hitables[0].radius == configs.WORLD_RADIUS
    mkinds = {desc.materials[i].kind for i in range(desc.n_materials)}
    assert {L.MATERIAL_SKY, L.MATERIAL_LAMBERTIAN, L.MATERIAL_DIELECTRIC, L.MATERIAL_EMISSIVE} <= mkinds
    # exact duplicate spheres (centre and radius) at different indices
    geo = {}
    for i in range(desc.n_hitables):
        h = desc.hitables[i]
        if h.kind == L.HITABLE_SPHERE:
            geo.setdefault(bytes(h)[8:24] + bytes(h)[52:64], []).append(i)
    assert sum(len(v) > 1 for v in geo.values()) >= 3
    # every light has its emissive sphere
    for k in range(desc.n_lights):
        l = desc.lights[k]
        h = desc.hitables[2 + k]
        assert list(h.center) == list(l.pos) and desc.materials[h.material].kind == L.MATERIAL_EMISSIVE
    # the same arguments give the same bytes, another seed other ones
    assert _flat(*configs.sphere_field((64, 48), 500, 64, 300, seed=3)[::-1])[1:] == (hit, mat, lig)
    assert _flat(*configs.sphere_field((64, 48), 500, 64, 300, seed=4)[::-1])[1] != hit


def test_sphere_field_places_the_fractal_and_moves_spheres():
    for at in (0, 7, 40):
        cam, w = configs.sphere_field((32, 32), 40, 4, 8, fractal_index=at)
        desc, _ = w.flatten(cam)
        assert [desc.hitables[i].kind for i in range(desc.n_hitables)].index(L.HITABLE_MANDELBOX) == min(at, 40)
    cam, w = configs.sphere_field((32, 32), 40, 4, 8, fractal=False, moving=True)
    desc, _ = w.flatten(cam)
    assert desc.n_hitables == 40
    assert any(any(desc.hitables[i].center_velocity) for i in range(desc.n_hitables))


def test_oracle_renders_a_1024_hitable_scene():
    from oracle import binding
    cam, w = configs.sphere_field((16, 16), 1023, 256, 1024)
    desc, _ = w.flatten(cam)
    assert desc.n_hitables == L.RAYN_MAX_HITABLES
    integ = configs.PathTracingIntegrator(1, 2)
    inp = FrameInputs(16, 16, 1, integ)
    o, info = binding.render(w, cam, inp, (16, 16), integ, TR)
    assert info["extend_rays"] > 0
    assert np.isfinite(o["color"]).all() and float(o["color"].sum() + o["background"].sum()) > 0
