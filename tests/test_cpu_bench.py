"""bench.py plumbing that can be checked without a GPU: workload construction, names, peaks fallback, clock-log parsing."""
import argparse
import importlib.util
import os

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_headline_workload_is_the_reference_backed_config_3_and_weak_scaling_multiplies_spp():
    b = _bench()
    assert b.HEADLINE_CONFIG == 3  # Mandelbox = the only fractal SDF rayn defines (SURVEY F1)
    c1 = b.build_workload(3, "weak", 1)
    assert c1["res"] == (1920, 1080) and c1["spp"] == 512 and c1["max_bounces"] == 8
    assert "mandelbox" in b.workload_name(c1, "weak", 1) and b.workload_name(c1, "weak", 1).startswith("cfg3 ")
    c8 = b.build_workload(3, "weak", 8)
    assert c8["spp"] == 4096 and "spp x8" in b.workload_name(c8, "weak", 8)
    c2 = b.build_workload(2, "weak", 1)
    assert b.workload_name(c2, "weak", 1) == "cfg2 Mandelbulb(authored) 1024x1024 128spp 4b"
    s8 = b.build_workload(5, "strong", 8)
    assert s8["res"] == (7680, 4320) and s8["spp"] == 1024 and "spp fixed" in b.workload_name(s8, "strong", 8)


def test_effective_cores_respects_affinity_and_cgroup_quota(monkeypatch):
    b = _bench()
    n, info = b.effective_cores()
    assert 1 <= n <= (os.cpu_count() or 1) and info["affinity"] >= n
    import builtins
    real_open = builtins.open

    def fake_open(path, *a, **k):
        if path == "/sys/fs/cgroup/cpu.max":
            import io
            return io.StringIO("400000 100000\n")
        return real_open(path, *a, **k)
    monkeypatch.setattr(builtins, "open", fake_open)
    monkeypatch.setattr(os, "sched_getaffinity", lambda pid: set(range(128)), raising=False)
    n, info = b.effective_cores()
    assert n == 4 and info["cgroup_quota"] == 4.0 and info["affinity"] == 128


def test_cpu_sample_runs_the_oracle_without_mapping_the_cuda_library():
    """The CPU arm (cpu_baseline / --impl reference) builds its inputs through librayn_hostinputs.so and renders with the
    oracle: librayn_b200.so must not be mapped by it (VERDICT r1: the reference arm listed the product .so)."""
    import subprocess
    import sys
    code = (
        "import sys, os; sys.path.insert(0, %r)\n"
        "import importlib.util\n"
        "spec = importlib.util.spec_from_file_location('bench', os.path.join(%r, 'bench.py')); b = importlib.util.module_from_spec(spec); spec.loader.exec_module(b)\n"
        "from rayn_b200.film import FrameInputs\n"
        "c = b.build_workload(1, 'weak', 1)\n"
        "inp = FrameInputs(c['res'][0], c['res'][1], c['samples'], c['integrator'])\n"
        "r, dt = b.cpu_sample(c, inp, 0.5)\n"
        "maps = open('/proc/self/maps').read()\n"
        "assert 'librayn_b200' not in maps, 'CUDA library mapped by the CPU arm'\n"
        "assert 'librayn_oracle' in maps and 'librayn_hostinputs' in maps\n"
        "assert r['value'] > 0 and r['cores'] >= 1 and r['tiles'] >= 1 and r['kind'] == 'port'\n"
        "print('ok', r['tiles_per_thread'])\n" % (ROOT, ROOT))
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True)
    assert out.returncode == 0 and "ok" in out.stdout, out.stdout + out.stderr


def test_kernel_source_sha_is_stable_and_keys_the_traffic_file():
    b = _bench()
    assert b.kernel_source_sha() == b.kernel_source_sha() and len(b.kernel_source_sha()) == 16


def test_peaks_reads_measured_file_or_falls_back(tmp_path, monkeypatch):
    b = _bench()
    v, src = b.peaks()
    assert v > 1000 and ("measured" in src or "fallback" in src)
    monkeypatch.setattr(b, "ROOT", str(tmp_path))
    v, src = b.peaks()
    assert v == 6650.0 and "fallback" in src


def test_clock_log_parsing(tmp_path):
    b = _bench()
    s = b.ClockSampler.__new__(b.ClockSampler)
    f = open(tmp_path / "c.csv", "w+")
    f.write("0, 1965, 1965, 812.5, 0x0000000000000004, Not Active, Not Active, Not Active, Active\n"
            "0, 1950, 1965, 990.1, 0x0000000000000004, Not Active, Not Active, Not Active, Active\n"
            "garbage line\n"
            "0, 1305, 1965, 1001.0, 0x0, Not Active, Active, Not Active, Not Active\n")
    s.f = f

    class P:
        def terminate(self):
            pass

        def wait(self, timeout=None):
            return 0

        def kill(self):
            pass
    s.p = P()
    out = s.stop()
    assert out["samples"] == 3 and out["sm_mhz"] == 1950.0 and out["sm_max_mhz"] == 1965.0
    assert out["reasons"] == ["hw_thermal_slowdown", "sw_power_cap"]


def test_dump_outputs_writes_every_film_plane_per_pixel(tmp_path, monkeypatch):
    """--dump-outputs: the film store (color | alpha | background | normal planes) as float32 arrays with one row per pixel;
    frames above DUMP_MAX_PIXELS are a seeded pixel sample, the same on every run, and the headline dump stays under 64 MiB."""
    import numpy as np
    import torch
    b = _bench()
    assert b.DUMP_MAX_PIXELS * 10 * 4 <= 64 << 20
    w, h = 40, 30
    npx = w * h
    store = torch.arange(10 * npx, dtype=torch.float32)
    s = store.numpy()
    want = {"color": s[:3 * npx].reshape(npx, 3), "alpha": s[3 * npx:4 * npx], "background": s[4 * npx:7 * npx].reshape(npx, 3),
            "normal": s[7 * npx:].reshape(npx, 3)}
    b.dump_outputs(str(tmp_path / "full"), store, w, h)
    assert sorted(os.listdir(tmp_path / "full")) == sorted(f"{k}.npy" for k in want)
    for k, v in want.items():
        got = np.load(tmp_path / "full" / f"{k}.npy")
        assert got.dtype == np.float32 and np.array_equal(got, v), k
    monkeypatch.setattr(b, "DUMP_MAX_PIXELS", 100)
    b.dump_outputs(str(tmp_path / "a"), store, w, h)
    b.dump_outputs(str(tmp_path / "b"), store, w, h)
    idx = np.sort(np.random.default_rng(0).choice(npx, 100, replace=False))
    for k, v in want.items():
        a = np.load(tmp_path / "a" / f"{k}.npy")
        assert np.array_equal(a, v[idx]) and np.array_equal(a, np.load(tmp_path / "b" / f"{k}.npy")), k


def test_committed_traffic_profile_belongs_to_this_kernel_build():
    """bench.py reports `roofline.traffic` only from an ncu capture of THIS kernel build: profiles/r02_traffic.json is keyed by the
    hash of the kernel sources.  A kernel edit without a new capture must be noticed (the line then says traffic: null)."""
    import json
    import bench
    tj = json.load(open(os.path.join(os.path.dirname(os.path.abspath(bench.__file__)), "profiles", "r02_traffic.json")))
    assert tj["kernel_source_sha"] == bench.kernel_source_sha(), "kernel sources changed after the last ncu capture: re-run tools/profile_r02.sh"
    for cfg in ("cfg3", "cfg2"):
        for k in ("k_extend_march", "k_shadow"):
            assert tj[cfg][k]["dram_bytes_per_launch"] > 0
