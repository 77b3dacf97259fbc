"""The C-ABI libraries load and export every symbol include/mcs.h declares (no GPU compute here)."""
import ctypes as C
import os
import re

import pytest

import mcs_b200
from mcs_b200 import abi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    txt = open(os.path.join(ROOT, "include", "mcs.h")).read()
    return sorted(set(re.findall(r"MCS_API\s+[\w\s\*]+?\b(mcs_\w+)\s*\(", txt)))


def test_header_and_mirror_agree():
    assert header_symbols() == sorted(abi.ABI_SYMBOLS)


def test_oracle_exports_abi(olib):
    for s in header_symbols():
        assert hasattr(olib, s)
    assert olib.mcs_backend().decode() == "cpu-oracle"


def test_cuda_library_exports_abi():
    p = mcs_b200.lib_path()
    assert os.path.exists(p), "libmcs_b200.so not built: run __graft_entry__.build()"
    lib = abi.bind(C.CDLL(p))  # also checks struct sizes against the ctypes mirror
    for s in header_symbols():
        assert hasattr(lib, s)
    assert lib.mcs_backend().decode() == "cuda-sm_100a"


def test_cuda_library_is_not_stale():
    """A failed nvcc build must not leave an older libmcs_b200.so in place unnoticed."""
    src = os.path.join(ROOT, "montecarloscattering.jl_b200", "csrc")
    newest = max(os.path.getmtime(os.path.join(src, f)) for f in os.listdir(src) if f.endswith((".cu", ".cuh")))
    newest = max(newest, os.path.getmtime(os.path.join(ROOT, "include", "mcs.h")))
    assert os.path.getmtime(mcs_b200.lib_path()) >= newest, "libmcs_b200.so is older than its sources: rebuild"


def test_default_config_identical(olib):
    lib = abi.bind(C.CDLL(mcs_b200.lib_path()))
    a, b = abi.default_config(olib), abi.default_config(lib)
    assert bytes(a) == bytes(b)
    assert a.helix_cap == 10_000 and a.xn_per_fine == 2000.0 and a.E_rel_pt == 0.005
    assert a.mp_g * a.c_cms == pytest.approx(5.01439438e-14, rel=1e-8)  # README.md:5 of the reference


def test_no_cpu_fallback_without_gpu():
    """Where no GPU is visible the product must fail loudly, never compute on the CPU.  Checked in a child process that sees
    no device (CUDA_VISIBLE_DEVICES empty), so that it also holds on a machine with GPUs."""
    import subprocess
    import sys
    code = ("import mcs_b200\nfrom mcs_b200 import abi\n"
            "lib = mcs_b200.load_cuda_library()\ncfg = abi.default_config(lib)\n"
            "cfg.n_grid, cfg.num_psd_mom_bins, cfg.num_psd_theta_bins = 99, 171, 159\n"
            "try:\n    abi.Engine(lib, cfg)\nexcept abi.McsError as e:\n    print(e)\n")
    out = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                         capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr
    assert "no CUDA device" in out.stdout, out.stdout


def test_package_does_not_import_oracle():
    pkg = os.path.join(ROOT, "montecarloscattering.jl_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dp, f)).read()
                assert "oracle_engine" not in txt and "mcs_oracle" not in txt, f


def test_plain_c_caller_builds_and_runs(tmp_path):
    """include/mcs.h from a C (not C++) translation unit of a third party: tests/c_caller.c is compiled with gcc -std=c99
    -pedantic-errors, linked against the CPU oracle (same ABI as the CUDA library) and run through one pcut."""
    import subprocess
    exe = tmp_path / "c_caller"
    odir = os.path.join(ROOT, "oracle")
    cc = subprocess.run(["gcc", "-std=c99", "-pedantic-errors", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
                         os.path.join(ROOT, "tests", "c_caller.c"), "-o", str(exe), "-L", odir, "-lmcs_oracle", "-lm",
                         f"-Wl,-rpath,{odir}"], capture_output=True, text=True)
    assert cc.returncode == 0, cc.stderr
    run = subprocess.run([str(exe)], capture_output=True, text=True, timeout=120)
    assert run.returncode == 0, run.stdout + run.stderr
    assert "c_caller ok: backend cpu-oracle" in run.stdout
