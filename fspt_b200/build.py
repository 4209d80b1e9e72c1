"""In-tree build of libfspt_b200.so (nvcc, sm_100a only).  `python -m fspt_b200.build`."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT_DIR = os.path.join(HERE, "lib")
LIB = os.path.join(OUT_DIR, "libfspt_b200.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")

# --fmad=false + IEEE div/sqrt + no FTZ: the kernels follow the reference's f32 operation order exactly
# (DESIGN.md section 4); -lineinfo for ncu source pages.
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo",
    "--fmad=false", "--prec-div=true", "--prec-sqrt=true", "--ftz=false",
    "-Xcompiler", "-fPIC,-ffp-contract=off,-O2,-mssse3", "-Xptxas", "-v",
]
CXX_FLAGS = ["-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-pthread"]


def sources():
    return [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC))]


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    inc = os.path.join(HERE, "..", "include", "fspt_b200.h")
    return any(os.path.getmtime(s) > t for s in sources() + [inc, os.path.abspath(__file__)])


def build(force=False, verbose=False, defines=(), out=None):
    """defines/out: build an A/B variant (e.g. defines=["-DTRACE_REFILL=24"], out="lib/variants/x.so")."""
    lib = LIB if out is None else os.path.join(HERE, out)
    if out is None and not force and not needs_build():
        return LIB
    os.makedirs(os.path.dirname(lib), exist_ok=True)
    tag = "" if out is None else "_" + os.path.basename(out).replace(".so", "")
    obj_cu = os.path.join(OUT_DIR, "fspt_api%s.o" % tag)
    obj_bvh = os.path.join(OUT_DIR, "bvh_device.o")
    host = ["bvh_builder", "atlas_packer"]
    objs = [os.path.join(OUT_DIR, h + ".o") for h in host]
    cmds = [[NVCC] + NVCC_FLAGS + list(defines) + ["-c", os.path.join(CSRC, "fspt_api.cu"), "-o", obj_cu]]
    cmds += [[NVCC] + NVCC_FLAGS + ["-c", os.path.join(CSRC, "bvh_device.cu"), "-o", obj_bvh]]
    cmds += [["g++"] + CXX_FLAGS + ["-c", os.path.join(CSRC, h + ".cpp"), "-o", o] for h, o in zip(host, objs)]
    cmds += [[NVCC, "-shared", "-o", lib, obj_cu, obj_bvh] + objs + ["-Xlinker", "--no-undefined", "-lpthread"]]
    for cmd in cmds:
        r = subprocess.run(cmd, capture_output=True, text=True)
        if verbose or r.returncode != 0:
            sys.stderr.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
        if r.returncode != 0:
            raise RuntimeError("build failed: " + " ".join(cmd))
        if cmd[0] == NVCC and "-c" in cmd and out is None and obj_cu in cmd:
            with open(os.path.join(OUT_DIR, "ptxas.log"), "w") as f:
                f.write(r.stderr)
    return lib


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
