"""Scene scripts: `setup()` restates reference src/setup.rs:46-169; `baseline_config(n)` builds
the five BASELINE.json configs (SURVEY §8d "Synthetic inputs").

Mandelbulb configs (2, 4, 5) use an AUTHORED SDF: the reference has no Mandelbulb
(SURVEY F1), so for those configs parity is only ever oracle <-> GPU, never vs rayn.
"""
from .scene import (BoxFold, CameraStore, Dielectric, Emissive, HitableStore, Lambertian, Linear, MandelBox, Mandelbulb,
                    MaterialStore, PathTracingIntegrator, PinholeCamera, Sky, Sphere, SphereFold, SphereLight, Srgb,
                    ThinLensCamera, TracedSDF, Vec3, VolumeParams, World)

WORLD_RADIUS = 100.0       # setup.rs:33
FRACTAL_ITERATIONS = 12    # setup.rs:44
FRAME_RATE = 24            # main.rs:47


def frame_time_range(frame=1):
    """main.rs:47-49,61-62: frame_start = frame / 24, shutter 1/24."""
    import numpy as np
    start = np.float32(frame) * (np.float32(1.0) / np.float32(FRAME_RATE))
    end = start + np.float32(1.0) / np.float32(24.0)
    return float(start), float(end)


def _lights_and_emitters(materials, hitables, lights):
    """setup.rs:91-122"""
    green = Srgb(1.5, 4.5, 3.0).normalized()
    blue = Srgb(1.5, 3.0, 4.5).normalized()
    blue_emissive = materials.add_material(Emissive.new_splat(blue * 3.0))
    green_emissive = materials.add_material(Emissive.new_splat(green * 3.0))
    light_pairs = [(Vec3(1.2, -1.2, 1.2), 0.15), (Vec3(-1.2, 1.2, 1.2), 0.15)]
    for pos, rad in light_pairs:
        green_pos = pos.copy()
        green_pos.v[1] *= -1.0
        lights.append(SphereLight(green_pos, rad, green * 40.0))
        lights.append(SphereLight(pos, rad, blue * 40.0))
        hitables.push(Sphere(green_pos, rad - 0.01, green_emissive))
        hitables.push(Sphere(pos, rad - 0.01, blue_emissive))
    lights.append(SphereLight(Vec3.zero(), 0.25, green * 20.0))
    hitables.push(Sphere(Vec3.zero(), 0.24, green_emissive))


def setup(resolution=(1280, 720), volume=True, fractal="mandelbox", camera="pinhole", bulb_iterations=8):
    """setup.rs:46-169 -> (CameraHandle, World).  Defaults reproduce the reference scene."""
    materials, hitables, lights = MaterialStore(), HitableStore(), []
    volume_params = VolumeParams(0.25, 0.035) if volume else VolumeParams(None, None)  # setup.rs:55-60
    sky = materials.add_material(Sky(Srgb(0.3, 0.4, 0.6), Srgb(0.2, 0.3, 0.6) * 0.05))  # :63-69
    hitables.push(Sphere(Vec3(0.0, 0.0, 0.0), WORLD_RADIUS, sky))                        # :71
    grey = materials.add_material(Dielectric.new_remap(Srgb(0.2, 0.2, 0.2), 0.6))        # :76
    if fractal == "mandelbox":
        sdf = MandelBox(FRACTAL_ITERATIONS, BoxFold(1.0), SphereFold(0.01, 1.9), -2.1)   # :84
    elif fractal == "mandelbulb":
        sdf = Mandelbulb(bulb_iterations, 8, 2.0)
    else:
        raise ValueError(fractal)
    hitables.push(TracedSDF(sdf, grey))                                                   # :78-86
    _lights_and_emitters(materials, hitables, lights)
    origin = Vec3(-0.45, 0.2, 2.0) * 2.25                                                 # :134
    if camera == "pinhole":
        cam = PinholeCamera(resolution, 60.0, origin, Vec3(0.0, 0.0, 0.0), Vec3(0.0, 1.0, 0.0))  # :129-141
    elif camera == "thinlens":
        # config 4 "DOF": aperture 0.05, focused on the fractal centre (stated here, BASELINE leaves it open)
        cam = ThinLensCamera(resolution, 60.0, 0.05, origin, Vec3(0.0, 0.0, 0.0), Vec3(0.0, 1.0, 0.0), Vec3(0.0, 0.0, 0.0))
    else:
        raise ValueError(camera)
    cameras = CameraStore()
    handle = cameras.add_camera(cam)
    return handle, World(hitables, lights, materials, cameras, volume_params)


def setup_single_sphere(resolution=(256, 256)):
    """BASELINE config 1 (SURVEY §8d cfg1): sky + one Dielectric sphere r=1 + one SphereLight."""
    materials, hitables, lights = MaterialStore(), HitableStore(), []
    sky = materials.add_material(Sky(Srgb(0.3, 0.4, 0.6), Srgb(0.2, 0.3, 0.6) * 0.05))
    hitables.push(Sphere(Vec3(0.0, 0.0, 0.0), WORLD_RADIUS, sky))
    grey = materials.add_material(Dielectric.new_remap(Srgb(0.2, 0.2, 0.2), 0.6))
    hitables.push(Sphere(Vec3(0.0, 0.0, 0.0), 1.0, grey))
    lights.append(SphereLight(Vec3(1.2, 1.2, 1.2), 0.15, Srgb(1.0, 1.0, 1.0) * 40.0))
    cam = PinholeCamera(resolution, 60.0, Vec3(-0.45, 0.2, 2.0) * 2.25, Vec3(0.0, 0.0, 0.0), Vec3(0.0, 1.0, 0.0))
    cameras = CameraStore()
    handle = cameras.add_camera(cam)
    return handle, World(hitables, lights, materials, cameras, VolumeParams(None, None))


def sphere_field(res, n_spheres, n_lights, n_materials, fractal=True, seed=0, fractal_index=1, volume=False, moving=False):
    """An authored, seeded scene in the style of setup.rs at any size -> (CameraHandle, World).

    Hitables: the setup.rs sky sphere first, then `n_spheres - 1` analytic spheres: one emissive sphere per SphereLight
    (as setup.rs:91-122 pairs them), a few EXACT duplicates of earlier ground spheres with another material (so the
    first-index-wins tie rule of hitable.rs:177-198 decides what is hit) and a ground of small spheres; with `fractal`
    the setup.rs Mandelbox goes in at insertion index `fractal_index` (clamped).  Materials: sky, the Mandelbox's grey
    Dielectric, one Emissive, then a seeded mix of Lambertian / Dielectric / Emissive up to `n_materials`.  `moving` gives
    every seventh ground sphere a centre velocity (a `Linear` centre).  All values are float32, drawn from
    numpy.random.default_rng(seed): the same arguments give the same scene bit for bit."""
    import numpy as np
    n_spheres, n_lights, n_materials = int(n_spheres), int(n_lights), int(n_materials)
    if n_spheres < 1 + n_lights:
        raise ValueError("n_spheres must hold the sky sphere and one emissive sphere per light")
    if n_materials < 3:
        raise ValueError("n_materials must hold the sky, the grey Dielectric and one Emissive")
    rng = np.random.default_rng(seed)
    f32 = np.float32

    def u(lo, hi, size=None):
        return (f32(lo) + (f32(hi) - f32(lo)) * rng.random(size, dtype=np.float32)).astype(np.float32)

    materials, hitables, lights = MaterialStore(), HitableStore(), []
    sky = materials.add_material(Sky(Srgb(0.3, 0.4, 0.6), Srgb(0.2, 0.3, 0.6) * 0.05))  # setup.rs:63-69
    grey = materials.add_material(Dielectric.new_remap(Srgb(0.2, 0.2, 0.2), 0.6))       # :76
    emissive = [materials.add_material(Emissive.new_splat(Srgb(1.5, 4.5, 3.0).normalized() * 3.0))]
    while len(materials.items) < n_materials:
        kind = int(rng.integers(0, 3))
        col = Srgb(*u(0.1, 0.9, 3))
        if kind == 0:
            materials.add_material(Lambertian(col))
        elif kind == 1:
            materials.add_material(Dielectric.new_remap(col, float(u(0.1, 0.9))))
        else:
            emissive.append(materials.add_material(Emissive.new_splat(col * 3.0)))
    spheres = [Sphere(Vec3(0.0, 0.0, 0.0), WORLD_RADIUS, sky)]  # setup.rs:71
    for k in range(n_lights):  # SphereLight + its emissive sphere, setup.rs:91-122
        pos = u(-1.0, 1.0, 3)
        pos = pos / np.sqrt(np.sum(pos * pos, dtype=np.float32), dtype=np.float32) * u(1.4, 2.4)
        rad = u(0.06, 0.15)
        lights.append(SphereLight(Vec3(*pos), float(rad), Srgb(*u(0.5, 1.0, 3)) * 30.0))
        spheres.append(Sphere(Vec3(*pos), float(rad - f32(0.01)), emissive[k % len(emissive)]))
    rest = n_spheres - 1 - n_lights
    n_dup = min(3, rest // 8)
    ground = []
    for i in range(rest - n_dup):
        r = u(0.04, 0.22)
        c = Vec3(float(u(-3.0, 3.0)), float(f32(-1.4) + r * f32(2.0) * u(0.0, 1.0)), float(u(-3.0, 3.0)))
        mat = int(rng.integers(1, n_materials))
        centre = Linear(c, Vec3(0.0, float(u(-0.5, 0.5)), 0.0)) if moving and i % 7 == 3 else c
        ground.append(Sphere(centre, float(r), mat))
    spheres += ground
    for d in range(n_dup):  # exact duplicates of earlier ground spheres, later in insertion order, another material
        src = ground[(d * 5) % len(ground)]
        dup = Sphere(Linear(Vec3(*src.center), Vec3(*src.center_velocity)), float(src.radius), (src.material % (n_materials - 1)) + 1)
        spheres.append(dup)
    if fractal:
        box = TracedSDF(MandelBox(FRACTAL_ITERATIONS, BoxFold(1.0), SphereFold(0.01, 1.9), -2.1), grey)  # setup.rs:78-86
        spheres.insert(max(0, min(int(fractal_index), len(spheres))), box)
    for h in spheres:
        hitables.push(h)
    cam = PinholeCamera(res, 60.0, Vec3(-0.45, 0.2, 2.0) * 2.25, Vec3(0.0, 0.0, 0.0), Vec3(0.0, 1.0, 0.0))  # setup.rs:129-141
    cameras = CameraStore()
    handle = cameras.add_camera(cam)
    volume_params = VolumeParams(0.25, 0.035) if volume else VolumeParams(None, None)  # setup.rs:55-60
    return handle, World(hitables, lights, materials, cameras, volume_params)


# name, resolution, SAMPLES (spp = 4x), max_bounces, builder kwargs
BASELINE_CONFIGS = {
    1: dict(name="cfg1-sphere-256x256-4spp-2b", res=(256, 256), samples=1, max_bounces=2, scene="sphere"),
    2: dict(name="cfg2-mandelbulb-1024x1024-128spp-4b", res=(1024, 1024), samples=32, max_bounces=4,
            scene=dict(volume=False, fractal="mandelbulb")),
    3: dict(name="cfg3-mandelbox-1920x1080-512spp-8b-nee", res=(1920, 1080), samples=128, max_bounces=8,
            scene=dict(volume=False, fractal="mandelbox")),
    4: dict(name="cfg4-mandelbulb-volume-dof-2048x2048-256spp-4b", res=(2048, 2048), samples=64, max_bounces=4,
            scene=dict(volume=True, fractal="mandelbulb", camera="thinlens")),
    5: dict(name="cfg5-mandelbulb-7680x4320-1024spp-8b", res=(7680, 4320), samples=256, max_bounces=8,
            scene=dict(volume=False, fractal="mandelbulb")),
}


def baseline_config(n, res=None, samples=None, max_bounces=None):
    """-> dict(name, res, samples, spp, integrator, camera, world).  res/samples/max_bounces override for downscaled tests."""
    c = dict(BASELINE_CONFIGS[n])
    if res is not None:
        c["res"] = tuple(res)
    if samples is not None:
        c["samples"] = samples
    if max_bounces is not None:
        c["max_bounces"] = max_bounces
    if c["scene"] == "sphere":
        cam, world = setup_single_sphere(c["res"])
    else:
        cam, world = setup(c["res"], **c["scene"])
    c["camera"], c["world"] = cam, world
    c["spp"] = 4 * c["samples"]
    c["integrator"] = PathTracingIntegrator(c["max_bounces"], 2)
    return c
