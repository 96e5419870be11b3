"""TEST INFRASTRUCTURE — host emulation of the CUDA sources.

Builds webrender_b200/csrc/wrcu_api.cu with plain g++ (-DWRCU_HOSTEMU, see
csrc/hostemu_shim.h) into tests/_build/libwrcu_emu.so with every C-ABI symbol
renamed wrcu_* → wremu_*.  The library runs the SAME per-instance (setup) and
per-pixel (shade) device functions as the kernels, in plain loops on the host,
so shader logic can be checked against the oracle on a box without a GPU.

It is never part of the product: nothing under webrender_b200/ loads it, and
parity claims rest on the real kernels (tests -m gpu).
"""
import ctypes as C
import os
import subprocess

from webrender_b200 import abi
from webrender_b200.device import DeviceBase, WrcuError, bind_prefixed

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "webrender_b200", "csrc")
LIB = os.path.join(ROOT, "tests", "_build", "libwrcu_emu.so")


def build():
    srcs = [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    if os.path.exists(LIB) and all(os.path.getmtime(s) <= os.path.getmtime(LIB) for s in srcs):
        return LIB
    os.makedirs(os.path.dirname(LIB), exist_ok=True)
    renames = [f"-D{s}={s.replace('wrcu_', 'wremu_', 1)}" for s in abi.SYMBOLS]
    # parallel test workers may build at once: each links its own file and renames it into place
    tmp = f"{LIB}.{os.getpid()}"
    cmd = ["g++", "-x", "c++", "-std=c++17", "-O1", "-fPIC", "-shared", "-ffp-contract=off", "-fno-math-errno",
           "-DWRCU_HOSTEMU", "-w"] + renames + ["-o", tmp, os.path.join(CSRC, "wrcu_api.cu"), "-lm"]
    subprocess.run(cmd, check=True)
    os.replace(tmp, LIB)
    return LIB


class EmuDevice(DeviceBase):
    prefix = "wremu_"

    def __init__(self):
        self.lib = C.CDLL(build())
        bind_prefixed(self.lib, "wremu_")
        self.lib.wremu_ctx_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        self.lib.wremu_ctx_destroy.argtypes = [C.c_void_p]
        self.lib.wremu_finish.argtypes = [C.c_void_p]
        ctx = C.c_void_p()
        rc = self.lib.wremu_ctx_create(0, C.byref(ctx))
        if rc:
            raise WrcuError(rc, "wremu_ctx_create")
        self.ctx = ctx

    def finish(self):
        self._check(self.lib.wremu_finish(self.ctx))

    def close(self):
        if self.ctx:
            self.lib.wremu_ctx_destroy(self.ctx)
            self.ctx = None
