"""The kernels of cudalibrarysamples_b200/csrc/spmv_generic_kernels.cuh, THE SAME SOURCE, compiled for the host with g++ on top of
tests/host_emulation/cuda_emulation.h (a real thread per lane, a barrier-based __shfl_down_sync, a locked atomicAdd) and loaded with
ctypes; exports emu_csr_generic / emu_coo_generic / emu_sell_generic (tests/host_emulation/emulate_generic.cpp)."""
import ctypes as C
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU_DIR = os.path.join(ROOT, "tests", "host_emulation")


def load():
    """Build tests/host_emulation/_build/libgeneric_emu.so when a source is newer, then load it."""
    out = os.path.join(EMU_DIR, "_build", "libgeneric_emu.so")
    srcs = [os.path.join(EMU_DIR, "emulate_generic.cpp"), os.path.join(EMU_DIR, "cuda_emulation.h"),
            os.path.join(ROOT, "cudalibrarysamples_b200", "csrc", "spmv_generic_kernels.cuh")]
    if not os.path.exists(out) or any(os.path.getmtime(s) > os.path.getmtime(out) for s in srcs):
        os.makedirs(os.path.dirname(out), exist_ok=True)
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-pthread", "-shared", "-fPIC", "-I" + EMU_DIR,
                               "-I" + os.path.join(ROOT, "cudalibrarysamples_b200", "csrc"), srcs[0], "-o", out])
    return C.CDLL(out)
