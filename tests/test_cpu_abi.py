"""The C-ABI library loads on a CPU-only box and exports every symbol include/rayn_b200.h
declares; struct layouts of the ctypes binding equal the C compiler's; no compute calls."""
import ctypes as C
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "rayn_b200.h")


def _ensure_built():
    from rayn_b200 import build
    build.build()


def test_every_declared_symbol_is_exported_and_bound():
    _ensure_built()
    from rayn_b200 import _lib as L
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    declared = set(re.findall(r"\b(rayn_b200_\w+)\s*\(", text))
    assert len(declared) >= 20
    lib = L.lib()
    assert declared == set(L.SYMBOLS), f"binding/header mismatch: {declared ^ set(L.SYMBOLS)}"
    for name in declared:
        assert hasattr(lib, name), f"librayn_b200.so does not export {name}"
    assert lib.rayn_b200_abi_version() == 2
    assert lib.rayn_b200_muladd_fused() == (1 if L.MULADD_FUSED else 0)


def test_all_library_variants_load_and_export_the_abi():
    """default (mul_add unfused = stock rayn build), _fma (fused) and the legacy TEST build export the same ABI; the
    host-inputs library exports the pure-CPU builders without pulling in the CUDA runtime."""
    _ensure_built()
    from rayn_b200 import _lib as L
    bdir = os.path.dirname(L.LIB_PATH)
    for name, fused in (("librayn_b200.so", 0), ("librayn_b200_fma.so", 1), ("librayn_b200_legacy.so", 0)):
        l = C.CDLL(os.path.join(bdir, name))
        for sym in L.SYMBOLS:
            assert hasattr(l, sym), f"{name} lacks {sym}"
        assert l.rayn_b200_muladd_fused() == fused
    h = C.CDLL(L.HOSTLIB_PATH)
    for sym in L.HOST_SYMBOLS:
        assert hasattr(h, sym)
    ldd = subprocess.run(["ldd", L.HOSTLIB_PATH], capture_output=True, text=True).stdout
    assert "cudart" not in ldd and "libcuda" not in ldd
    ldd = subprocess.run(["ldd", L.LIB_PATH], capture_output=True, text=True).stdout
    assert "nccl" not in ldd, "NCCL must be resolved with dlopen at the first comm call, not at load time"


def test_struct_layouts_match_the_c_compiler(tmp_path):
    from rayn_b200 import _lib as L
    names = ["RaynHitable", "RaynMaterial", "RaynLight", "RaynCamera", "RaynVolume", "RaynRenderConsts", "RaynSceneDesc",
             "RaynFrameDesc", "RaynFilmPlanes", "RaynConfig", "RaynStats"]
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include "rayn_b200.h"\nint main(){' +
                   "".join(f'printf("{n} %zu\\n", sizeof({n}));' for n in names) +
                   'printf("off_scramble %zu\\n", offsetof(RaynFrameDesc, scramble));'
                   'printf("off_camera %zu\\n", offsetof(RaynSceneDesc, camera));return 0;}')
    exe = tmp_path / "sz"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    for n in names:
        assert C.sizeof(getattr(L, n)) == int(out[n]), n
    assert L.RaynFrameDesc.scramble.offset == int(out["off_scramble"])
    assert L.RaynSceneDesc.camera.offset == int(out["off_camera"])


def test_create_fails_loudly_without_a_gpu():
    """In a process that sees no device (CUDA_VISIBLE_DEVICES empty), so that it holds on a machine with a GPU too."""
    code = ("import sys; sys.path.insert(0, %r)\n"
            "from rayn_b200 import _lib as L\n"
            "from rayn_b200.film import Renderer\n"
            "try:\n"
            "    Renderer(0)\n"
            "except L.RaynError as e:\n"
            "    assert e.code == L.RAYN_ERR_NO_DEVICE, e.code\n"
            "    assert 'no CPU fallback' in str(e), str(e)\n"
            "    print('raised')\n" % ROOT)
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout.strip() == "raised", r.stdout + r.stderr


def test_product_never_touches_the_oracle():
    pkg = os.path.join(ROOT, "rayn_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h", ".hpp")):
                txt = open(os.path.join(dirpath, f), errors="ignore").read()
                for line in txt.splitlines():
                    s = line.strip()
                    if s.startswith(("import ", "from ", "#include")) and "oracle" in s:
                        raise AssertionError(f"{f}: product code references oracle/: {s}")
