"""Build tests/emu/libwbk_emu.so: the csrc/*.cu kernels compiled by g++ against the SIMT
emulation shim (TEST INFRASTRUCTURE ONLY -- never loaded by the product package).

build(variant="sinf_worst") builds tests/emu/libwbk_emu_sinf_worst.so instead, in which __sinf carries the
largest error CUDA documents for it (simt_emu.h, WBK_EMU_SINF_WORST)."""

import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
CSRC = os.path.join(ROOT, "wavebreaking_b200", "csrc")
LIB = os.path.join(HERE, "libwbk_emu.so")
VARIANTS = {None: [], "sinf_worst": ["-DWBK_EMU_SINF_WORST"]}


def build(force=False, variant=None):
    defs = VARIANTS[variant]
    suffix = "" if variant is None else "_" + variant
    lib = os.path.join(HERE, "libwbk_emu" + suffix + ".so")
    srcs = sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cu"))
    deps = srcs + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cuh")]
    deps += [os.path.join(HERE, "simt_emu.h"), os.path.join(HERE, "simt_emu.cpp"),
             os.path.join(ROOT, "include", "wbk.h")]
    if not force and os.path.exists(lib) and all(os.path.getmtime(d) <= os.path.getmtime(lib) for d in deps):
        return lib
    objs = []
    for s in srcs + [os.path.join(HERE, "simt_emu.cpp")]:
        o = os.path.join(HERE, "_obj" + suffix + "_" + os.path.basename(s) + ".o")
        cmd = ["g++", "-O1", "-g", "-std=c++17", "-fPIC", "-DWBK_EMU", *defs, "-ffp-contract=off",
               "-Wno-unused-result", "-x", "c++", "-include", os.path.join(HERE, "simt_emu.h"), "-I", CSRC, "-c", s,
               "-o", o]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError("emu build failed:\n" + " ".join(cmd) + "\n" + res.stderr[-6000:])
        objs.append(o)
    res = subprocess.run(["g++", "-shared", "-o", lib] + objs, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("emu link failed:\n" + res.stderr[-4000:])
    return lib


if __name__ == "__main__":
    print(build(force=True))
