"""In-tree build of libvbnmf.so (CUDA, sm_100a).  nvcc cross-compiles without a GPU.

    python -m ccfindr_b200.build [--force] [--verbose]

One translation unit for the host side and C ABI (csrc/vbnmf.cu) and one per padded rank
(csrc/rp_inst.cu with -DVB_RP=<RP>), compiled in parallel and linked into
ccfindr_b200/libvbnmf.so.  Objects are rebuilt only when a source they include changed.
"""
import concurrent.futures as cf
import hashlib
import os
import re
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(CSRC, "_obj" + os.environ.get("VBNMF_OBJ_SUFFIX", ""))
INCLUDE = os.path.join(HERE, "..", "include")
LIB = os.path.join(HERE, os.environ.get("VBNMF_LIB_NAME", "libvbnmf.so"))  # experiments: variants

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "-I", INCLUDE]
if os.environ.get("VBNMF_SWEEP_THREADS"):  # tuning experiments only
    NVCC_FLAGS.append("-DVB_SWEEP_THREADS=" + os.environ["VBNMF_SWEEP_THREADS"])
if os.environ.get("VBNMF_LPN_BYTES"):
    NVCC_FLAGS.append("-DVB_LPN_BYTES=" + os.environ["VBNMF_LPN_BYTES"])
if os.environ.get("VBNMF_SWEEP_THREADS_F32"):
    NVCC_FLAGS.append("-DVB_SWEEP_THREADS_F32=" + os.environ["VBNMF_SWEEP_THREADS_F32"])
if os.environ.get("VBNMF_MID_THREADS"):
    NVCC_FLAGS.append("-DVB_MID_THREADS=" + os.environ["VBNMF_MID_THREADS"])
if os.environ.get("VBNMF_MID_THREADS_COLS"):
    NVCC_FLAGS.append("-DVB_MID_THREADS_COLS=" + os.environ["VBNMF_MID_THREADS_COLS"])
if os.environ.get("VBNMF_WIDE_THREADS"):
    NVCC_FLAGS.append("-DVB_WIDE_THREADS=" + os.environ["VBNMF_WIDE_THREADS"])
if os.environ.get("VBNMF_UNROLL"):
    NVCC_FLAGS.append("-DVB_UNROLL=" + os.environ["VBNMF_UNROLL"])
if os.environ.get("VBNMF_SPLIT_PRED"):
    NVCC_FLAGS.append("-DVB_SPLIT_PRED=" + os.environ["VBNMF_SPLIT_PRED"])
if os.environ.get("VBNMF_SKIP_DEAD"):
    NVCC_FLAGS.append("-DVB_SKIP_DEAD=" + os.environ["VBNMF_SKIP_DEAD"])
if os.environ.get("VBNMF_DOT_CHAINS"):
    NVCC_FLAGS.append("-DVB_DOT_CHAINS=" + os.environ["VBNMF_DOT_CHAINS"])
for _d in os.environ.get("VBNMF_DEFS", "").split():   # experiments: "VB_X=1 VB_Y=0" -> -DVB_X=1 ...
    if _d.startswith("VB_"):
        NVCC_FLAGS.append("-D" + _d)
if os.environ.get("VBNMF_LP_BITS"):   # count bits of the log-product bound term (kernels.cuh)
    NVCC_FLAGS.append("-DVB_LP_BITS=" + os.environ["VBNMF_LP_BITS"])


def _nvcc():
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def ranks():
    txt = open(os.path.join(CSRC, "rp_ranks.h")).read()
    return [int(v) for v in re.findall(r"F\((\d+)\)", txt)]


def _source_hash():
    hsh = hashlib.sha256()
    files = sorted(os.listdir(CSRC)) + [os.path.join(INCLUDE, "vbnmf.h")]
    for f in files:
        p = f if os.path.isabs(f) else os.path.join(CSRC, f)
        if os.path.isfile(p) and p.endswith((".cu", ".cuh", ".h")):
            hsh.update(f.encode())
            hsh.update(open(p, "rb").read())
    hsh.update(" ".join(NVCC_FLAGS).encode())
    return hsh.hexdigest()


def kernel_hash():
    """Hash of the sweep / update kernel sources (profiles/traffic.json is stamped with it: an ncu
    capture describes the kernels it was taken from; the host side, vbnmf.cu, does not enter)."""
    hsh = hashlib.sha256()
    for f in ("kernels.cuh", "kernels_common.cuh", "special.cuh", "rp_inst.cu", "rp_table.h",
              "rp_ranks.h"):
        hsh.update(f.encode())
        hsh.update(open(os.path.join(CSRC, f), "rb").read())
    hsh.update(" ".join(a for a in NVCC_FLAGS if a.startswith("-DVB_")).encode())
    return hsh.hexdigest()[:16]


def _run(cmd, verbose):
    if verbose:
        print(" ".join(cmd), flush=True)
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("build failed: %s\n%s\n%s" % (" ".join(cmd), res.stdout, res.stderr))
    return res.stdout + res.stderr


def build(force=False, verbose=False, jobs=None):
    os.makedirs(OBJ, exist_ok=True)
    stamp = os.path.join(OBJ, "stamp.txt")
    want = _source_hash()
    if (not force and os.path.exists(LIB) and os.path.exists(stamp)
            and open(stamp).read().strip() == want):
        return LIB
    nvcc = _nvcc()
    units = [("vbnmf.o", ["-c", os.path.join(CSRC, "vbnmf.cu")])]
    for rp in ranks():
        units.append(("rp_inst_%d.o" % rp, ["-DVB_RP=%d" % rp, "-c", os.path.join(CSRC, "rp_inst.cu")]))
    objs = []
    jobs = jobs or max(1, (os.cpu_count() or 2))
    with cf.ThreadPoolExecutor(max_workers=jobs) as ex:
        futs = []
        for name, args in units:
            out = os.path.join(OBJ, name)
            objs.append(out)
            futs.append(ex.submit(_run, [nvcc] + NVCC_FLAGS + args + ["-o", out], verbose))
        for f in futs:
            f.result()
    _run([nvcc, "-shared", "-o", LIB] + objs + ["-lcudart", "-ldl", "-lpthread"], verbose)
    with open(stamp, "w") as f:
        f.write(want)
    return LIB


if __name__ == "__main__":
    lib = build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print(lib)
