"""Speed of the scene-table path (scenes beyond 16 hitables / materials / lights).  Prints ONE JSON line:

  sweep:   Msamples/s of configs.sphere_field at 1920x1080, Mandelbox on, 4 lights, 8 materials, 4 bounces, for 14, 17, 64,
           256 and 1024 hitables (14: the parameter-block path, 17: the first scene-table one), at a spp that makes every
           frame last >= 1 s, plus the per-kernel shares of one RAYN_FLAG_TIMING frame;
  paths:   BASELINE configs 3 and 2 at full size through the parameter block and through the tables
           (RAYN_FLAG_SCENE_TABLES), alternated frame by frame, with their spread.

Times are the library's device events around each render call (RaynStats.total_ms); inputs and film stay on the device.
The card's name and power limit are read in the same run.  Usage: python tools/bench_scene_size.py [--reps N] [--out FILE]
"""
import argparse
import json
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from rayn_b200 import _lib as L  # noqa: E402
from rayn_b200 import configs  # noqa: E402
from rayn_b200.dist import device_frame_desc  # noqa: E402
from rayn_b200.film import FrameInputs, Renderer  # noqa: E402

TR = configs.frame_time_range(1)
SWEEP = (14, 17, 64, 256, 1024)


class Frame:
    """One scene, one frame geometry, device-resident inputs and film; render() returns (Msamples/s, ms, stats)."""

    def __init__(self, cam, world, res, samples, integrator, flags=0):
        w, h = res
        inp = FrameInputs(w, h, samples, integrator)
        self.dev = [torch.from_numpy(a).cuda() for a in inp.arrays()]
        self.store = torch.zeros(10 * w * h, dtype=torch.float32, device="cuda")
        npx = w * h
        s = self.store
        self.planes = L.RaynFilmPlanes(s[:3 * npx].data_ptr(), s[3 * npx:4 * npx].data_ptr(), s[4 * npx:7 * npx].data_ptr(), s[7 * npx:].data_ptr(),
                                       L.MEM_DEVICE)
        self.desc = device_frame_desc(self.dev, w, h, (16, 16), samples, integrator, 1, TR, (inp.sets_1d, inp.sets_2d))
        self.r = Renderer(0, flags=flags)
        self.r.upload_scene(world, cam)
        torch.cuda.synchronize()

    def render(self):
        self.r.render(self.desc, self.planes)
        st = self.r.stats()
        return st.paths / (st.total_ms * 1e-3) / 1e6, st.total_ms, st

    def close(self):
        self.r.close()


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clk = [x.strip() for x in q.stdout.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit": power, "sm_max_clock": clk}


def spread(v):
    m = sum(v) / len(v)
    return {"mean": m, "min": min(v), "max": max(v), "spread_pct": 100.0 * (max(v) - min(v)) / m, "values": v}


def sweep_point(n_hit, reps):
    integ = configs.PathTracingIntegrator(4, 2)
    cam, world = configs.sphere_field((1920, 1080), n_hit - 1, 4, 8, seed=0)
    cal = Frame(cam, world, (1920, 1080), 1, integ)
    cal.render()
    _, ms, _ = cal.render()
    cal.close()
    samples = max(1, math.ceil(1600.0 / ms))  # >= 1 s per frame: ms is for SAMPLES = 1 (4 spp), and frame time grows less than linearly in spp
    timed = Frame(cam, world, (1920, 1080), 1, integ, flags=L.FLAG_TIMING)
    timed.render()
    _, _, st = timed.render()
    tot = sum(st.kernel_ms[k] for k in range(L.STAT_KERNELS))
    shares = {L.KERNEL_NAMES[k]: round(100.0 * st.kernel_ms[k] / tot, 2) for k in range(L.STAT_KERNELS) if st.kernel_ms[k] > 0}
    timed.close()
    f = Frame(cam, world, (1920, 1080), samples, integ)
    f.render()
    vals, mss = [], []
    for _ in range(reps):
        v, ms, _ = f.render()
        vals.append(v)
        mss.append(ms)
    f.close()
    return {"hitables": n_hit, "path": "tables" if n_hit > 16 else "parameter block", "samples": samples, "spp": 4 * samples,
            "ms_per_frame": sum(mss) / len(mss), "msamples_per_s": spread(vals), "kernel_shares_pct": shares}


def paths_point(cfg, reps):
    c = configs.baseline_config(cfg)
    frames = {name: Frame(c["camera"], c["world"], c["res"], c["samples"], c["integrator"], flags) for name, flags in
              (("parameter_block", 0), ("tables", L.FLAG_SCENE_TABLES))}
    vals = {name: [] for name in frames}
    for f in frames.values():
        f.render()
    for _ in range(reps):
        for name, f in frames.items():  # alternated
            vals[name].append(f.render()[0])
    films = [f.store for f in frames.values()]
    same = bool(torch.equal(films[0].view(torch.int32), films[1].view(torch.int32)))
    for f in frames.values():
        f.close()
    return {"config": c["name"], "films_bit_identical": same, **{k: spread(v) for k, v in vals.items()}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    out = {"what": "scene-size sweep (sphere_field) and parameter-block vs scene-table path on configs 3 and 2", "unit": "Msamples/s",
           "card": card(), "sweep": [sweep_point(n, args.reps) for n in SWEEP],
           "paths": [paths_point(3, args.reps), paths_point(2, 2 * args.reps)]}
    out["card_after"] = card()
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
