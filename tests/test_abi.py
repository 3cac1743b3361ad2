"""CPU tier: the C-ABI libraries load, export every symbol their headers declare, and refuse to run without a GPU."""
import ctypes as C
import importlib
import os
import re
import subprocess
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared(header):
    text = open(os.path.join(REPO, "include", header)).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(drt_[a-z0-9_]+)\s*\(", text)))


def test_cuda_library_exports_header(drt):
    cuda = importlib.import_module("daily-ray-trace_b200.cuda")
    L = cuda.lib()
    names = _declared("drt_cuda.h")
    assert len(names) >= 12
    for name in names:
        assert hasattr(L, name), name
    assert set(cuda.EXPORTS) == set(names)


def test_host_library_exports_header(host):
    L = host.lib()
    for name in _declared("drt_host.h"):
        assert hasattr(L, name), name


def test_no_cpu_fallback_without_device():
    """Run where no device is visible (a child process with CUDA_VISIBLE_DEVICES empty, so that this holds on a GPU machine too)."""
    code = ("import importlib, sys\n"
            "cuda = importlib.import_module('daily-ray-trace_b200.cuda')\n"
            "assert cuda.device_count() == 0\n"
            "try:\n"
            "    cuda.Context(0)\n"
            "except cuda.CudaError as e:\n"
            "    sys.exit(0 if e.code == -101 else 3)\n"
            "sys.exit(2)\n")
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    run = subprocess.run([sys.executable, "-c", code], cwd=REPO, env=env, capture_output=True, text=True)
    assert run.returncode == 0, (run.returncode, run.stderr[-2000:])
