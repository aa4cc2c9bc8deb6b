"""TEST INFRASTRUCTURE: builds tests/host_emu/_build/libgfr_emu.so (g++, host only)."""
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
OUT_DIR = os.path.join(HERE, "_build")
OUT = os.path.join(OUT_DIR, "libgfr_emu.so")
DEPENDS = [os.path.join(HERE, "gfr_emu.cpp"),
           os.path.join(ROOT, "grid-fed-rl-gym_b200", "csrc", "gfr_device.cuh"),
           os.path.join(ROOT, "grid-fed-rl-gym_b200", "csrc", "gfr_image.hpp"),
           os.path.join(ROOT, "include", "gfr_b200.h")]


def build() -> str:
    os.makedirs(OUT_DIR, exist_ok=True)
    if os.path.exists(OUT) and all(os.path.getmtime(d) <= os.path.getmtime(OUT) for d in DEPENDS):
        return OUT
    cmd = ["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=fast", "-pthread",
           # the header-only builder is also compiled into libgfr_b200.so, which loads with RTLD_GLOBAL: without these
           # the emulation would bind to THAT copy of the inline functions (stale whenever the two are built apart)
           "-fvisibility-inlines-hidden", "-Wl,-Bsymbolic",
           # the CTA-wide groups' paths (row pipeline, packed pool-child records) on the 8- and 16-lane teams, the
           # warp-sized groups' ones on the 2- and 4-lane teams
           "-DGFR_WIDE_GROUP_MIN_LANES=8", "-o", OUT,
           os.path.join(HERE, "gfr_emu.cpp"), "-lm"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("g++ failed:\n" + res.stdout + res.stderr)
    return OUT


if __name__ == "__main__":
    print(build())
