#!/usr/bin/env python
"""bench.py — Msamples/s (pixels x spp) of the wavefront render path on B200.

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
  python bench.py --impl reference --gpus N --steps K ...  # CPU restatement of rayn's path (oracle) on the host cores

A "step" is one full `render_frame_into` of the workload.  The headline workload is BASELINE config 3 — the Mandelbox
scene of the reference's own setup.rs at 1920x1080, 512 spp, 8 bounces + NEE: the largest 1-GPU config and the only fractal
config whose SDF exists in rayn (configs 2/4/5 use an authored Mandelbulb, SURVEY F1).  The same JSON line carries, under
"also", config 2 (1-GPU Mandelbulb config) and config 5 (the 8K Mandelbulb config, strong-scaled: fixed 7680x4320x1024spp
frame over the N GPUs) so that the driver's 1/2/4/8 runs yield a cfg5 strong-scaling curve with a 1-GPU denominator.

At N>1 film tiles are sharded `(tile_x + tile_y) % N == rank` through the C ABI (`rayn_b200_render_frame_sharded`: no
data-path collective; one NCCL all-gather of the film at the end of each step, inside the timed region, issued by the
library on its render stream).  The headline is weak-scaled (spp x N, per-GPU work fixed); `--scaling strong` keeps the
config fixed instead.  After the timed loop rank 0 re-renders a few tiles alone and compares them BITWISE with the gathered
film (`parity`); a mismatch exits non-zero.

`value` is measured with the sampler tables, scramble plane and film resident in HBM; `e2e` goes through the public
host-buffer API (H2D of the inputs and D2H of the film planes inside the timed region).  One JSON line on stdout (rank 0).
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the tree may be read-only: the bench leaves nothing in it

import numpy as np  # noqa: E402

ALG_BYTES_EXTEND = 40.0   # SURVEY §8(d): K2 reads float4 o+time, float4 d+closest (32 B), writes t+key (8 B)
ALG_BYTES_SHADOW = 36.0   # K5 reads seg_a + seg_b (32 B), clears at most one visibility bit (4 B)
ALG_BYTES_SHADE = 184.0   # shade: read ray 68 + hit 8, write ray 68 or film <= 40
ALG_BYTES_RAYGEN = 88.0   # writes o_time, d_t, rad, thr, nrm0 (5 x float4) + term + q_live per path
ALG_BYTES_RESOLVE = 36.0  # reads rad + nrm0 (2 x float4) + term per path (+ 40 B per pixel out)
MANDELBULB_FLOP_PER_ITER = 75.0  # authored formula, counted in DESIGN.md §4
MANDELBOX_FLOP_PER_ITER = 25.0   # SURVEY §8(d)
FLOP_PER_EVAL_TAIL = 10.0
# non-tensor FP32 peak: MEASURED FFMA rate (profiles/r02_ubench_pipes.txt: 243.0 lane-flop/clk/SM) x 148 SMs x max clock
FP32_PEAK_TFLOPS = 148 * 243.0 * 1.965e9 / 1e12
HEADLINE_CONFIG = 3


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=HEADLINE_CONFIG)
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--res", type=int, nargs=2, default=None, help="override resolution (debug)")
    ap.add_argument("--samples", type=int, default=None, help="override SAMPLES (spp/4) (debug)")
    ap.add_argument("--cpu-seconds", type=float, default=25.0, help="target wall time of one CPU sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-also", action="store_true", help="skip the secondary configs (2 and 5) reported under 'also'")
    ap.add_argument("--max-paths", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the film planes of the last timed step of the headline workload to DIR/<plane>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def kernel_source_sha():
    """Identifies the kernel build a profile belongs to (profiles/*_traffic.json are keyed by it)."""
    h = hashlib.sha256()
    for f in ("rt_kernels.cuh", "rt_sdf2.cuh", "rt_device.cuh", "detmath.h", "api.cu"):
        h.update(open(os.path.join(ROOT, "rayn_b200", "csrc", f), "rb").read())
    return h.hexdigest()[:16]


def effective_cores():
    """Host cores this process may actually use: CPU affinity AND the cgroup CPU quota (a 1-GPU lease of a 128-thread
    box is typically capped at 16 CPUs by cpu.max while os.cpu_count() still says 128)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    quota = None
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            quota = float(q) / float(p)
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            p = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / p
        except Exception:
            pass
    eff = n if quota is None else max(1, min(n, int(quota + 0.5)))
    return eff, {"os_cpu_count": os.cpu_count(), "affinity": n, "cgroup_quota": quota}


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1]))
                mx.append(float(c[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        return out


DUMP_MAX_PIXELS = 1 << 20  # 10 float32 channels per pixel: at most 40 MiB per dump


def dump_outputs(out_dir, store, w, h):
    """The film a caller of the timed path receives, as float32 arrays with one row per pixel (row-major, y up):
    color.npy and background.npy and normal.npy [n, 3], alpha.npy [n].  A frame of more than DUMP_MAX_PIXELS pixels is
    sampled: pixels np.sort(np.random.default_rng(0).choice(w * h, DUMP_MAX_PIXELS, replace=False)), the same for every
    run at that resolution, so that two builds can be compared output for output."""
    import torch
    npx = w * h
    if npx > DUMP_MAX_PIXELS:
        idx = np.sort(np.random.default_rng(0).choice(npx, DUMP_MAX_PIXELS, replace=False))
    else:
        idx = np.arange(npx)
    sel = torch.from_numpy(idx).to(store.device)
    os.makedirs(out_dir, exist_ok=True)
    off = 0
    for name, ch in (("color", 3), ("alpha", 1), ("background", 3), ("normal", 3)):
        a = store[off * npx:(off + ch) * npx].view(npx, ch).index_select(0, sel).cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), a if ch > 1 else a[:, 0])
        off += ch


def build_workload(cfgnum, scaling, world, res=None, samples=None):
    from rayn_b200 import configs
    base = configs.BASELINE_CONFIGS[cfgnum]
    if samples is None:
        samples = base["samples"]
    if scaling == "weak" and world > 1:
        samples *= world
    c = configs.baseline_config(cfgnum, res=res, samples=samples)
    c["time_range"] = configs.frame_time_range(1)
    c["cfgnum"] = cfgnum
    return c


def workload_name(c, scaling, world):
    w, h = c["res"]
    s = f"{c['name'].split('-')[0]} {'Mandelbulb(authored)' if 'mandelbulb' in c['name'] else c['name'].split('-')[1]} {w}x{h} {c['spp']}spp {c['max_bounces']}b"
    if world > 1:
        s += f" tiles (tx+ty)%{world} ({scaling}: spp {'x' + str(world) if scaling == 'weak' else 'fixed'})"
    return s


# ---------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle (C++ SSE-packet restatement of rayn's path, OpenMP over tiles like rayon) on the host cores
# ---------------------------------------------------------------------------------------------------------------
def cpu_sample(c, inputs, target_seconds):
    """Time the CPU oracle on every k-th tile of the workload.  Threads = the cores this process can really use
    (affinity and cgroup quota).  The sample holds >= 16 tiles per thread whenever that fits ~4x the time target, so the
    wall-clock figure is not tail-bound; otherwise (very expensive tiles: weak-scaled spp) the balanced figure
    samples / (process CPU seconds / threads) is reported instead, which charges the CPU arm no tail at all."""
    from oracle import binding as ob
    from rayn_b200.film import tile_grid
    w, h = c["res"]
    n_tiles = int(np.prod(tile_grid(w, h, 16, 16)))
    threads, core_info = effective_cores()

    def run(k):
        t0, c0 = time.perf_counter(), time.process_time()
        _, info = ob.render(c["world"], c["camera"], inputs, (16, 16), c["integrator"], c["time_range"], n_threads=threads, subsample_k=k)
        return time.perf_counter() - t0, time.process_time() - c0, info["tiles"]

    # probe: ~2 tiles per thread spread over the frame
    k = max(1, n_tiles // max(2 * threads, 8))
    dt, ct, tiles = run(k)
    per_tile_cpu = ct / max(tiles, 1)
    want = max(16 * threads, int(target_seconds * threads / max(per_tile_cpu, 1e-9)))
    if want * per_tile_cpu / threads > 4.0 * target_seconds:  # 16 tiles per thread do not fit the time budget
        want = max(2 * threads, int(target_seconds * threads / max(per_tile_cpu, 1e-9)))
    want = min(n_tiles, want)
    k2 = max(1, n_tiles // want)
    if k2 != k:
        dt, ct, tiles = run(k2)
        k = k2
    samples_done = tiles * 256 * c["spp"]
    tiles_per_thread = tiles / threads
    wall_value = samples_done / dt / 1e6
    balanced_value = samples_done / (ct / threads) / 1e6
    use_wall = tiles_per_thread >= 16
    return dict(value=wall_value if use_wall else balanced_value, unit="Msamples/s", cores=threads, cores_effective=threads, kind="port",
                timing="wall clock" if use_wall else "balanced: samples / (process CPU seconds / threads) — fewer than 16 tiles per thread fit the time budget",
                wall_value=wall_value, balanced_value=balanced_value, tiles=tiles, tiles_per_thread=tiles_per_thread, seconds=dt, core_info=core_info,
                sample=f"every {k}-th 16x16 tile of the workload ({tiles} of {n_tiles} tiles, {samples_done / 1e6:.2f} Msamples, {dt:.1f} s wall, "
                       f"{threads} OpenMP threads = affinity/cgroup allotment), OpenMP over tiles like rayon; C++ SSE-packet restatement of "
                       f"rayn's path, `wide` mul_add unfused like a stock cargo build (rayn itself cannot be built here: no Rust toolchain)"), dt


def run_reference(args, rank, world):
    """--impl reference: the CPU restatement of rayn's render path on the host cores.  Touches neither the GPU nor
    librayn_b200.so (frame inputs come from librayn_hostinputs.so).  Whatever --steps says, the arm makes TWO bounded
    samples of the workload (one if --steps 1), each >= 16 tiles per thread when that fits ~60 s, and reports their mean and
    their spread: a CPU "step" of the full frame would take 15-20 minutes, and many short samples would each be tail-bound."""
    if rank != 0:
        return
    from rayn_b200.film import FrameInputs
    from oracle import binding as ob
    ob.build()
    c = build_workload(args.config, args.scaling, world, args.res, args.samples)
    w, h = c["res"]
    inputs = FrameInputs(w, h, c["samples"], c["integrator"])
    n = 2 if args.steps >= 2 else 1
    vals, secs, last = [], 0.0, None
    for _ in range(n):
        last, dt = cpu_sample(c, inputs, min(args.cpu_seconds, 30.0))
        vals.append(last["value"])
        secs += dt
    v = float(np.mean(vals))
    last["value"] = v
    last["run_to_run"] = {"values": vals, "spread_rel": float((max(vals) - min(vals)) / max(v, 1e-12)), "samples_taken": n}
    line = {"impl": "reference", "metric": "Msamples/sec (pixels x spp)", "value": v, "unit": "Msamples/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": secs / n * 1e3, "higher_is_better": True,
            "scaling": args.scaling if world > 1 else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(c, args.scaling, world), "bounded_sample": True,
                       "steps_note": f"{n} bounded samples regardless of --steps (see cpu_baseline.sample); ms_per_step = mean sample time"},
            "cpu_baseline": last, "e2e": {"value": v, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------------
class Bench:
    def __init__(self, args, rank, world, local_rank):
        import torch
        self.torch, self.args, self.rank, self.world, self.local_rank = torch, args, rank, world, local_rank
        self.dev = torch.device("cuda", local_rank)

    def barrier(self):
        if self.world > 1:
            self.torch.distributed.barrier()
        self.torch.cuda.synchronize()

    def allmax(self, x):
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.torch.distributed.all_reduce(t, op=self.torch.distributed.ReduceOp.MAX)
        return float(t.item())

    def allsum(self, x):
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.torch.distributed.all_reduce(t, op=self.torch.distributed.ReduceOp.SUM)
        return float(t.item())

    def run_config(self, cfgnum, scaling, steps, warmup, breakdown=True, e2e=True, parity_tiles=6, dump_dir=None):
        """One workload: resident-input `value`, per-kernel breakdown, e2e, N>1 parity.  Returns a dict (all ranks).
        With `dump_dir`, rank 0 writes the film of the last timed step there before anything else renders into it."""
        torch = self.torch
        from rayn_b200 import _lib as L
        from rayn_b200.dist import DistFilm, device_frame_desc
        from rayn_b200.film import FrameInputs, Renderer, make_frame_desc, tile_grid
        args, rank, world = self.args, self.rank, self.world
        c = build_workload(cfgnum, scaling, world, args.res if cfgnum == args.config else None, args.samples if cfgnum == args.config else None)
        w, h = c["res"]
        tile = (16, 16)
        inputs = FrameInputs(w, h, c["samples"], c["integrator"])
        sets = (inputs.sets_1d, inputs.sets_2d)
        inputs_dev = [torch.from_numpy(a).to(self.dev) for a in inputs.arrays()]
        r = Renderer(self.local_rank, max_paths_per_pass=args.max_paths)
        r.upload_scene(c["world"], c["camera"])
        film = DistFilm(r, w, h, tile, rank, world)
        fdesc = device_frame_desc(inputs_dev, w, h, tile, c["samples"], c["integrator"], 1, c["time_range"], sets)

        def step_resident():
            film.render_gathered(fdesc)  # 1 GPU: render_frame; N GPUs: render_frame_sharded (shard render + NCCL film gather)

        for _ in range(warmup):
            step_resident()
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        launches, lib_ms = 0, 0.0
        t0 = time.perf_counter()
        e0.record()
        for _ in range(steps):
            step_resident()
            st = r.stats()
            launches += st.launches
            lib_ms += st.total_ms
        e1.record()
        torch.cuda.synchronize()
        wall_ms = (time.perf_counter() - t0) * 1e3
        ev_ms = e0.elapsed_time(e1)
        self.barrier()
        if dump_dir is not None and rank == 0:
            dump_outputs(dump_dir, film.store, w, h)
        st = r.stats()
        total_samples = self.allsum(float(st.paths))
        ms_per_step = self.allmax(max(ev_ms, lib_ms)) / steps
        out = {"workload": workload_name(c, scaling, world), "value": total_samples / (ms_per_step * 1e-3) / 1e6, "unit": "Msamples/s",
               "ms_per_step": ms_per_step, "steps": steps, "warmup": warmup, "samples_total": int(total_samples), "gpu_launches": int(launches),
               "passes_per_step": int(st.passes), "wall_ms_per_step": wall_ms / steps, "scaling": scaling if world > 1 else "weak",
               "timing": {"library_event_ms_per_step": lib_ms / steps, "host_event_ms_per_step": ev_ms / steps,
                          "rule": "max over ranks of max(device time inside the library calls, host-side event bracket), / steps"}}

        # ---- N > 1: the gathered film against a single-GPU re-render of sampled tiles, bit for bit --------------------
        if world > 1:
            ok, k = True, 0
            if rank == 0:
                ntx, nty = tile_grid(w, h, *tile)
                fr = [(0.5, 0.5), (0.4, 0.55), (0.62, 0.45), (0.05, 0.9), (0.33, 0.37), (0.7, 0.62), (0.48, 0.52), (0.55, 0.4)][:max(parity_tiles, world)]
                tiles = sorted({int(fx * ntx) * nty + int(fy * nty) for fx, fy in fr} | {i * nty + (world - 1 - i) % nty for i in range(min(world, ntx))})
                solo = torch.zeros(10 * w * h, dtype=torch.float32, device=self.dev)
                npx = w * h
                sp = L.RaynFilmPlanes(solo[:3 * npx].data_ptr(), solo[3 * npx:4 * npx].data_ptr(), solo[4 * npx:7 * npx].data_ptr(),
                                      solo[7 * npx:].data_ptr(), L.MEM_DEVICE)
                r2 = Renderer(self.local_rank, max_paths_per_pass=args.max_paths)
                r2.upload_scene(c["world"], c["camera"])
                sdesc = device_frame_desc(inputs_dev, w, h, tile, c["samples"], c["integrator"], 1, c["time_range"], sets, tiles)
                r2.render(sdesc, sp)
                r2.close()
                gathered = film.store.view(torch.int32)
                alone = solo.view(torch.int32)
                mask = torch.zeros(h, w, dtype=torch.bool, device=self.dev)
                owners = set()
                for idx in tiles:
                    x0, y0 = (idx // nty) * 16, (idx % nty) * 16
                    mask[y0:y0 + 16, x0:x0 + 16] = True
                    owners.add(((idx // nty) + (idx % nty)) % world)
                m1 = mask.reshape(-1)
                m3 = m1.repeat_interleave(3)
                full_mask = torch.cat([m3, m1, m3, m3])
                ok = bool(torch.equal(gathered[full_mask], alone[full_mask])) and bool((solo[full_mask] != 0).any())
                k = len(tiles)
                out["parity"] = {"tiles": k, "bit_identical": ok, "ranks_covered": len(owners),
                                 "what": "gathered N-GPU film vs the same tiles rendered by rank 0 alone, all 10 channel floats, bitwise"}
                del solo
            ok = self.allmax(0.0 if ok else 1.0) == 0.0
            out["parity_ok"] = ok

        # ---- per-kernel breakdown + roofline (separate TIMING context so events do not perturb `value`) ------------
        if breakdown:
            rt = Renderer(self.local_rank, max_paths_per_pass=args.max_paths, flags=L.FLAG_TIMING)
            rt.upload_scene(c["world"], c["camera"])
            # same device film, no second communicator: times this rank's shard only
            tdesc = device_frame_desc(inputs_dev, w, h, tile, c["samples"], c["integrator"], 1, c["time_range"], sets, film.tile_list)
            rt.render(tdesc, film.planes)
            rt.render(tdesc, film.planes)
            ts = rt.stats()
            out["kernels"], out["roofline"] = self.kernel_report(c, ts, w, h)
            rt.close()

        # ---- e2e: host buffers through the public API, H2D + D2H inside the timed region ---------------------------
        if e2e:
            pin = [torch.from_numpy(a).pin_memory() for a in inputs.arrays()]
            npx = w * h
            out_pin = torch.zeros(10 * npx, dtype=torch.float32).pin_memory()
            hp = L.RaynFilmPlanes(out_pin.data_ptr(), out_pin[3 * npx:].data_ptr(), out_pin[4 * npx:].data_ptr(), out_pin[7 * npx:].data_ptr(), L.MEM_HOST)
            hdesc = make_frame_desc(w, h, tile, c["samples"], c["integrator"], 1, c["time_range"], tuple(t.data_ptr() for t in pin), L.MEM_HOST, 0, 1, sets)
            h2d = sum(t.numel() * 4 for t in pin)
            d2h = out_pin.numel() * 4
            e2e_steps = min(steps, 5)  # a full host round trip per step; 5 are enough for a wall-clock mean
            film.render_gathered(hdesc, hp)
            self.barrier()
            t0 = time.perf_counter()
            chk = 0.0
            for _ in range(e2e_steps):
                film.render_gathered(hdesc, hp)  # returns after the film planes are in host memory
                chk += float(out_pin[0]) + float(out_pin[3 * npx - 1])
            dt = time.perf_counter() - t0
            self.barrier()
            dt = self.allmax(dt)
            out["e2e"] = {"value": total_samples / (dt / e2e_steps) / 1e6, "unit": "Msamples/s", "steps": e2e_steps, "h2d_bytes_per_step": int(h2d) * world,
                          "d2h_bytes_per_step": int(d2h) * world, "per_rank": {"h2d": int(h2d), "d2h": int(d2h)},
                          "timing": "host wall clock around the public host-buffer call (rayn_b200_render_frame / _sharded), max over ranks"}
            del pin, out_pin
        self._cpu_ctx = (c, inputs)
        r.close()
        del film, inputs_dev
        torch.cuda.empty_cache()
        return out

    def kernel_report(self, c, ts, w, h):
        from rayn_b200 import _lib as L
        kms = {L.KERNEL_NAMES[i]: float(ts.kernel_ms[i]) for i in range(len(L.KERNEL_NAMES)) if ts.kernel_launches[i]}
        klaunch = {L.KERNEL_NAMES[i]: int(ts.kernel_launches[i]) for i in range(len(L.KERNEL_NAMES)) if ts.kernel_launches[i]}
        ksum = sum(kms.values())
        hbm_peak, peak_src = peaks()
        is_bulb = "mandelbulb" in c["name"]
        sdf = [hh for hh in c["world"].hitables.items if hasattr(hh, "sdf")]
        iters = sdf[0].sdf.iterations if sdf else 0

        def flops(evals, bulb_iters):  # algorithmic flops of `evals` distance evaluations, from the iterations ACTUALLY run
            if is_bulb:
                return MANDELBULB_FLOP_PER_ITER * bulb_iters + FLOP_PER_EVAL_TAIL * evals
            return (MANDELBOX_FLOP_PER_ITER * iters + FLOP_PER_EVAL_TAIL) * evals

        per = {k: {"ms": kms[k], "share": kms[k] / max(ksum, 1e-9), "launches": klaunch[k]} for k in kms}
        ext_s, shd_s = kms.get("extend", 0.0) * 1e-3, kms.get("shadow", 0.0) * 1e-3
        if "extend" in per:
            per["extend"].update(rays=int(ts.extend_rays), sdf_evals=int(ts.sdf_evals_extend),
                                 iterations_per_eval=(ts.bulb_iters_extend / max(ts.sdf_evals_extend, 1)) if is_bulb else iters,
                                 march_slots_busy=ts.sdf_evals_extend / max(64.0 * ts.march_trips_extend, 1.0),
                                 hbm_gbs_algorithmic=ts.extend_rays * ALG_BYTES_EXTEND / max(ext_s, 1e-12) / 1e9,
                                 fp32_tflops_algorithmic=flops(ts.sdf_evals_extend, ts.bulb_iters_extend) / max(ext_s, 1e-12) / 1e12)
        if "shadow" in per:
            n_seg = int(ts.shadow_rays)  # light samples prepared; the segments actually marched are fewer (exact pre-filters)
            per["shadow"].update(shadow_rays=n_seg, sdf_evals=int(ts.sdf_evals_shadow),
                                 iterations_per_eval=(ts.bulb_iters_shadow / max(ts.sdf_evals_shadow, 1)) if is_bulb else iters,
                                 march_slots_busy=ts.sdf_evals_shadow / max(64.0 * ts.march_trips_shadow, 1.0),
                                 hbm_gbs_algorithmic=n_seg * ALG_BYTES_SHADOW / max(shd_s, 1e-12) / 1e9,
                                 fp32_tflops_algorithmic=flops(ts.sdf_evals_shadow, ts.bulb_iters_shadow) / max(shd_s, 1e-12) / 1e12)
        if "normals" in per:
            per["normals"].update(sdf_evals=int(ts.sdf_evals_normals))
        if "shade_pre" in per:
            shade_s = (kms.get("shade_pre", 0.0) + kms.get("shade_post", 0.0)) * 1e-3
            per["shade_pre"].update(lanes=int(ts.shade_lanes), hbm_gbs_algorithmic_pre_plus_post=ts.shade_lanes * ALG_BYTES_SHADE / max(shade_s, 1e-12) / 1e9)
        if "raygen" in per:
            per["raygen"]["hbm_gbs_algorithmic"] = ts.paths * ALG_BYTES_RAYGEN / max(kms["raygen"] * 1e-3, 1e-12) / 1e9
            per["raygen"]["hbm_frac"] = per["raygen"]["hbm_gbs_algorithmic"] / hbm_peak
        if "resolve" in per:
            per["resolve"]["hbm_gbs_algorithmic"] = (ts.paths * ALG_BYTES_RESOLVE + w * h * 40.0) / max(kms["resolve"] * 1e-3, 1e-12) / 1e9
            per["resolve"]["hbm_frac"] = per["resolve"]["hbm_gbs_algorithmic"] / hbm_peak
        dom = max(kms, key=kms.get) if kms else "extend"
        dom_name = {"extend": "k_extend_march (closest-hit sphere-march, sdf.rs:59-83)", "shadow": "k_shadow (occlusion sphere-march, sdf.rs:25-57)",
                    "shade_pre": "k_shade_pre", "shade_post": "k_shade_post"}.get(dom, dom)
        achieved = per[dom].get("hbm_gbs_algorithmic", 0.0)
        roofline = {"kernel": dom_name, "bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                    "peak_source": peak_src, "traffic": None,
                    "launches_of_kernel_per_step": klaunch.get(dom, 0), "avg_launch_ms": kms.get(dom, 0.0) / max(klaunch.get(dom, 1), 1),
                    "note": "the march kernels are FP32-pipe bound, not HBM bound (SURVEY F7: ~40 B and 1e4-1e5 flop per ray): `achieved` is the "
                            "contract's algorithmic bytes / kernel time and is small by construction; the roof that binds is reported in `fp32`",
                    "fp32": {"peak_tflops": FP32_PEAK_TFLOPS, "peak_source": "measured FFMA issue rate, profiles/r02_ubench_pipes.txt (243 lane-flop/clk/SM x 148 SMs x 1965 MHz)",
                             "extend_tflops": per.get("extend", {}).get("fp32_tflops_algorithmic"),
                             "extend_frac": per.get("extend", {}).get("fp32_tflops_algorithmic", 0.0) / FP32_PEAK_TFLOPS,
                             "shadow_tflops": per.get("shadow", {}).get("fp32_tflops_algorithmic"),
                             "shadow_frac": per.get("shadow", {}).get("fp32_tflops_algorithmic", 0.0) / FP32_PEAK_TFLOPS,
                             "flop_model": "SURVEY §8(d): Mandelbox 25 flop x iterations + 10 per evaluation (div, sqrt = 1); Mandelbulb 75 x iterations "
                                           "ACTUALLY RUN (counted by the kernels) + 10"}}
        # measured DRAM traffic of the dominant kernel: only from an ncu capture of THIS kernel build (keyed by source hash)
        tpath = os.path.join(ROOT, "profiles", "r02_traffic.json")
        if os.path.exists(tpath):
            tj = json.load(open(tpath))
            key = {"extend": "k_extend_march", "shadow": "k_shadow"}.get(dom)
            ent = tj.get(f"cfg{c['cfgnum']}", {}).get(key) if key else None
            if ent and tj.get("kernel_source_sha") == kernel_source_sha():
                roofline["traffic"] = ent["dram_bytes_per_launch"]
                roofline["traffic_note"] = ent.get("note", "") + f" (source: {ent.get('source', '?')})"
        return per, roofline


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return 0

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the rayn_b200 path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    b = Bench(args, rank, world, local_rank)

    clocks = ClockSampler(local_rank) if rank == 0 else None  # started before warm-up (nvidia-smi needs ~0.3 s to emit its first line)
    main_res = b.run_config(args.config, args.scaling, args.steps, args.warmup, breakdown=True, e2e=not args.no_e2e, dump_dir=args.dump_outputs)
    clock_info = clocks.stop() if clocks else None
    cpu_ctx = b._cpu_ctx

    also = {}
    if not args.no_also and args.res is None and args.samples is None:
        if args.config != 2 and world == 1:
            r2 = b.run_config(2, "weak", 3, 2, breakdown=True, e2e=not args.no_e2e)
            also["cfg2"] = {k: r2[k] for k in ("workload", "value", "unit", "ms_per_step", "steps", "warmup", "e2e", "gpu_launches", "roofline", "kernels") if k in r2}
            also["cfg2"]["note"] = "BASELINE config 2 (1 GPU): authored Mandelbulb, no rayn counterpart (SURVEY F1)"
        if args.config != 5:
            # one untimed step first: pass buffers (25 GB) are allocated lazily.  Per-kernel breakdown only at N > 1 (two more frames)
            r5 = b.run_config(5, "strong", 1, 1, breakdown=world > 1, e2e=False)
            also["cfg5_strong"] = {k: r5[k] for k in ("workload", "value", "unit", "ms_per_step", "steps", "warmup", "gpu_launches", "parity", "passes_per_step", "scaling", "kernels") if k in r5}
            also["cfg5_strong"]["note"] = ("BASELINE config 5 (7680x4320 Mandelbulb, 1024 spp, 8 bounces), the FIXED frame tiled across the N GPUs of this run: "
                                           "value(N) / value(1) over the driver's 1/2/4/8 runs is the strong-scaling curve; one timed step after one untimed step (a step is tens of seconds at N = 1)")
            if not r5.get("parity_ok", True):
                main_res["parity_ok"] = False

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu, _ = cpu_sample(cpu_ctx[0], cpu_ctx[1], args.cpu_seconds)

    parity_ok = main_res.get("parity_ok", True)
    if rank == 0:
        line = {"metric": "Msamples/sec (pixels x spp)", "value": main_res["value"], "unit": "Msamples/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": main_res["ms_per_step"], "higher_is_better": True, "scaling": main_res["scaling"],
                "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": main_res["workload"], "tile": "16x16", "samples_total": main_res["samples_total"],
                           "l2": "working set (path state >= 3 GB/pass) far exceeds the 126 MB L2; no explicit flush",
                           "mul_add": "unfused (stock `cargo run --release` rayn; oracle/README.md A6)",
                           "parallelism": f"dp{world}: 16x16 film tiles, (tx+ty)%{world} interleave, ncclAllGather of the film inside the library" if world > 1 else "1 GPU"},
                "clocks": clock_info, "e2e": main_res.get("e2e"), "gpu_launches": main_res["gpu_launches"], "roofline": main_res.get("roofline"),
                "cpu_baseline": cpu, "kernels": main_res.get("kernels"), "wall_ms_per_step": main_res["wall_ms_per_step"],
                "passes_per_step": main_res["passes_per_step"], "also": also, "kernel_source_sha": kernel_source_sha()}
        if "parity" in main_res:
            line["parity"] = main_res["parity"]
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0 if parity_ok else 3


if __name__ == "__main__":
    sys.exit(main())
