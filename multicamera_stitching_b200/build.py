"""In-tree build of ``libmcs_b200.so`` (the C-ABI library, sm_100a only).

``python -m multicamera_stitching_b200.build`` or ``__graft_entry__.build()``.
nvcc cross-compiles without a GPU; the resulting ``.so`` lives next to this
file so it travels with the source tree.
"""
import os
import shutil
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
REPO_DIR = os.path.dirname(PKG_DIR)
CSRC_DIR = os.path.join(PKG_DIR, "csrc")
LIB_PATH = os.path.join(PKG_DIR, "libmcs_b200.so")

SOURCES = ["mcs_plan.cu", "mcs_tiles.cu", "mcs_stitch.cu", "mcs_stitch_tiled.cu", "mcs_stitch_weighted.cu", "mcs_stitch_multiband.cu", "mcs_seams.cu", "mcs_seams_graphcut.cu", "mcs_exposure.cu", "mcs_match.cu", "mcs_ransac.cu", "mcs_resize.cu", "mcs_hostio.cu", "mcs_refit.cu"]
HEADERS = [os.path.join(CSRC_DIR, "mcs_common.h"), os.path.join(CSRC_DIR, "mcs_device.cuh"),
           os.path.join(REPO_DIR, "include", "mcs.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "--fmad=false",                      # the coordinate recipe must not be contracted
    "-Xcompiler", "-fPIC,-O2,-ffp-contract=off",
    "-Xptxas", "-v",
    "-I", os.path.join(REPO_DIR, "include"),
    "-I", CSRC_DIR,
]


def find_nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (set $NVCC)")


def is_stale():
    if not os.path.exists(LIB_PATH):
        return True
    built = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC_DIR, s) for s in SOURCES] + HEADERS + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > built for d in deps)


def build(force=False, verbose=False):
    """Compile the library if any source is newer than it; returns its path."""
    if not force and not is_stale():
        return LIB_PATH
    nvcc = find_nvcc()
    objs = []
    procs = []
    os.makedirs(os.path.join(PKG_DIR, "build"), exist_ok=True)
    for s in SOURCES:
        obj = os.path.join(PKG_DIR, "build", s.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + ["-c", os.path.join(CSRC_DIR, s), "-o", obj]
        procs.append((s, cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
        objs.append(obj)
    log = []
    for s, cmd, p in procs:
        out = p.communicate()[0].decode(errors="replace")
        log.append("$ " + " ".join(cmd) + "\n" + out)
        if p.returncode != 0:
            raise RuntimeError("nvcc failed on %s:\n%s" % (s, out))
    link = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB_PATH] + objs
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
    log.append("$ " + " ".join(link) + "\n" + r.stdout.decode(errors="replace"))
    if r.returncode != 0:
        raise RuntimeError("link failed:\n" + r.stdout.decode(errors="replace"))
    with open(os.path.join(PKG_DIR, "build", "build.log"), "w") as f:
        f.write("\n".join(log))
    if verbose:
        sys.stdout.write("\n".join(log) + "\n")
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
