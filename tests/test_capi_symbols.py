"""CPU-only checks of the drop-in boundary: the C-ABI library loads without a GPU and exports every
symbol that include/basic_dsp_b200.h declares (no compute calls here)."""
import ctypes
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "basic_dsp_b200.h")


def declared_functions():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    src = re.sub(r"^\s*#.*$", "", src, flags=re.M)
    src = re.sub(r"typedef[^;]*;", "", src)
    # `T name(args) BDSP_SYMBOL("sym");` declares the exported symbol `sym` (names that clash with glibc's <math.h>)
    src = re.sub(r"\b[A-Za-z_][A-Za-z0-9_]*(\s*\([^;{}()]*\))\s*BDSP_SYMBOL\(\s*\"([A-Za-z0-9_]+)\"\s*\)\s*;", r"\2\1;", src)
    names = re.findall(r"\b([A-Za-z_][A-Za-z0-9_]*)\s*\([^;{}]*\)\s*;", src)
    return sorted({n for n in names if not n.startswith("Bdsp") and n not in ("defined", "__asm__")})


@pytest.fixture(scope="module")
def libpath():
    import basic_dsp_b200
    if not os.path.exists(basic_dsp_b200.LIB_PATH):
        from basic_dsp_b200 import build
        build.build()
    return basic_dsp_b200.LIB_PATH


def test_header_declares_the_hot_path_surface():
    names = declared_functions()
    for s in ("32", "64"):
        for base in ("new", "delete_vector", "plain_fft", "plain_ifft", "fft", "ifft", "convolve_signal", "convolve",
                     "convolve_real", "convolve_complex", "multiply_frequency_response", "interpolatef",
                     "interpolatef_custom", "interpolate_lin", "real_scale", "complex_scale", "mul", "magnitude", "phase",
                     "get_magnitude", "get_phase", "get_mag_phase", "swap_halves", "zero_interleave", "to_complex",
                     "overwrite_data", "data", "complex_data", "clone"):
            assert base + s in names, base + s
    assert len(names) > 150


def test_library_exports_every_declared_symbol(libpath):
    lib = ctypes.CDLL(libpath)
    missing = [n for n in declared_functions() if not hasattr(lib, n)]
    assert not missing, missing


def test_no_undeclared_c_symbols_leak(libpath):
    out = subprocess.run(["nm", "-D", "--defined-only", libpath], capture_output=True, text=True).stdout
    exported = {l.split()[-1] for l in out.splitlines() if " T " in l}
    declared = set(declared_functions())
    extra = {e for e in exported if not e.startswith("_Z")} - declared
    assert not extra, extra


def test_python_binding_declares_prototypes_without_gpu(libpath):
    import basic_dsp_b200 as bd
    L = bd.lib()
    assert b"sm_100a" in L.bdsp_version()
    assert bd.device_count() >= 0
    assert bd.kernel_launch_count() == 0 or bd.device_count() > 0


def test_no_cpu_fallback_without_device(libpath):
    import numpy as np
    import basic_dsp_b200 as bd
    if bd.device_count() > 0:
        pytest.skip("a CUDA device is present")
    with pytest.raises(bd.DspError):
        bd.DspVec(np.ones(8, dtype=np.complex64))


def test_product_does_not_import_the_oracle():
    pkg = os.path.join(ROOT, "basic_dsp_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".hpp")):
                text = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in text.replace("no CPU fallback", ""), os.path.join(dirpath, f)


def test_every_cuda_source_is_built():
    from basic_dsp_b200 import build
    on_disk = {f for f in os.listdir(build.CSRC) if f.endswith(".cu")}
    assert on_disk == set(build.SOURCES), (sorted(on_disk - set(build.SOURCES)), sorted(set(build.SOURCES) - on_disk))


def test_one_build_one_code_path():
    """The shipped kernels are the only kernels: no build switches, no environment overrides in the CUDA sources."""
    from basic_dsp_b200 import build
    offenders = []
    for f in sorted(os.listdir(build.CSRC)):
        if f.endswith((".cu", ".cuh")):
            for i, line in enumerate(open(os.path.join(build.CSRC, f)), 1):
                if "getenv" in line or re.match(r"\s*#\s*(if|ifdef|ifndef|elif)\b", line):
                    offenders.append("%s:%d: %s" % (f, i, line.strip()))
    assert not offenders, offenders


def _build_cpp(tmp_path, libpath):
    exe = str(tmp_path / "host_mirror")
    src = os.path.join(ROOT, "tests", "cpp", "host_mirror.cpp")
    cmd = ["g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"), src, "-o", exe,
           "-L", os.path.dirname(libpath), "-lbasic_dsp_b200", "-Wl,-rpath," + os.path.dirname(libpath)]
    subprocess.check_call(cmd)
    return exe


def test_cpp_host_mirror_compiles_and_links(tmp_path, libpath):
    exe = _build_cpp(tmp_path, libpath)
    out = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stdout + out.stderr


@pytest.mark.gpu
def test_cpp_host_mirror_runs_on_gpu(tmp_path, libpath):
    exe = _build_cpp(tmp_path, libpath)
    out = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0 and "roundtrip" in out.stdout, out.stdout + out.stderr


def _build_c_example(tmp_path, libpath):
    exe = str(tmp_path / "c_example")
    src = os.path.join(ROOT, "examples", "c_example.c")
    cmd = ["gcc", "-std=c11", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), src, "-o", exe,
           "-L", os.path.dirname(libpath), "-lbasic_dsp_b200", "-Wl,-rpath," + os.path.dirname(libpath), "-lm"]
    subprocess.check_call(cmd)
    return exe


def test_header_is_valid_c11_and_the_c_example_links(tmp_path, libpath):
    """include/basic_dsp_b200.h is a C header (the reference's ABI is consumed from C, C#, Python ...)."""
    _build_c_example(tmp_path, libpath)


@pytest.mark.gpu
def test_c_example_runs_on_gpu(tmp_path, libpath):
    exe = _build_c_example(tmp_path, libpath)
    out = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0 and "spectrum peak" in out.stdout, out.stdout + out.stderr
    # cos(0.001 n) over 2^16 points: energy next to DC, which fft32 places at the centre bin
    idx = int(out.stdout.split("at bin")[1].split()[0])
    assert abs(idx - 32768) <= 12
