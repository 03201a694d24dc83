"""ctypes front-end of tests/emu/emu_table.cpp: the host emulator with the result-table user constraints.

TEST HARNESS ONLY.  TableEmulator / TableEmuEngine are emu_binding.Emulator / EmuEngine on a build of the emulator whose
residual, Jacobian, pair and sharded-range evaluations also run the table jobs (gelato_b200/csrc/user_table.h, DESIGN.md
section 10 "a16") as the CUDA library launches k_user_table; every entry point keeps its name and arguments.
"""
import ctypes
import os
import subprocess

import emu_binding

LIB = os.path.join(emu_binding.BUILD, "libgelato_emu_table.so")


def build(force=False):
    src = os.path.join(emu_binding._HERE, "emu", "emu_table.cpp")
    csrc = os.path.join(emu_binding.ROOT, "gelato_b200", "csrc")
    deps = [src, os.path.join(emu_binding._HERE, "emu", "emu.cpp"), os.path.join(emu_binding.ROOT, "include", "gelato_b200.h")] + [
        os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith((".h", ".inc"))]
    if not force and os.path.exists(LIB) and all(os.path.getmtime(LIB) >= os.path.getmtime(f) for f in deps):
        return LIB
    os.makedirs(emu_binding.BUILD, exist_ok=True)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-mfma", "-pthread", "-o", LIB, src])
    return LIB


class _TableLibrary:
    """Swaps the emulator library for this build after emu_binding has declared its prototypes."""

    def __init__(self, plan, scenario_plans=None):
        super().__init__(plan, scenario_plans=scenario_plans)
        base, self.L = self.L, ctypes.CDLL(build())
        for name in dir(base):
            if name.startswith("emu_"):
                f, g = getattr(self.L, name), getattr(base, name)
                f.argtypes, f.restype = g.argtypes, g.restype


class TableEmulator(_TableLibrary, emu_binding.Emulator):
    pass


class TableEmuEngine(_TableLibrary, emu_binding.EmuEngine):
    pass
