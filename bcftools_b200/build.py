"""In-tree build of the CUDA library (sm_100a only).  `python -m bcftools_b200.build`."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "lib", "libmcall_b200.so")
SOURCES = ["mcall_kernels.cu", "mcall_groups.cu", "mcall_biallelic.cu", "mcall_biallelic_groups.cu", "mcall_multi.cu", "mcall_triallelic.cu", "mcall_multi_warp.cu", "mcall_generic.cu", "mcall_abi.cu", "mcall_job.cu", os.path.join("host", "b200_call.c"), os.path.join("host", "b200_bcf.c"), os.path.join("host", "b200_driver.c"), os.path.join("host", "b200_vcf.c"), os.path.join("host", "b200_vcfcall.c"), os.path.join("host", "b200_pv4.c"), os.path.join("host", "b200_bcfio.c")]
HEADERS = ["mcall_kernels.cuh", "mcall_device.cuh", "mcall_multi.cuh", os.path.join(ROOT, "include", "mcall_b200.h"), os.path.join(ROOT, "include", "b200_call.h"), os.path.join(ROOT, "include", "mcall_job.h"), os.path.join(ROOT, "include", "b200_bcf.h"), os.path.join(ROOT, "include", "b200_driver.h"), os.path.join(ROOT, "include", "b200_vcf.h"), os.path.join(ROOT, "include", "b200_vcfcall.h"), os.path.join(ROOT, "include", "b200_bcfio.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "--fmad=false",   # no FMA contraction: the reference's x86-64 -O2 build has none
              "-I", os.path.join(ROOT, "include"), "-I", CSRC]


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES] + [h if os.path.isabs(h) else os.path.join(CSRC, h) for h in HEADERS]
    deps.append(os.path.abspath(__file__))
    return any(os.path.getmtime(d) > t for d in deps)


def _compile_link(out_path, extra, verbose=False, incremental=False):
    """One nvcc per source in parallel (objects under lib/obj/<name of the library>/), then one link.
    incremental: objects newer than their source, every header and this file are kept."""
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    objdir = os.path.join(os.path.dirname(LIB), "obj", os.path.basename(out_path))
    os.makedirs(objdir, exist_ok=True)
    hdrs = [h if os.path.isabs(h) else os.path.join(CSRC, h) for h in HEADERS] + [os.path.abspath(__file__)]
    procs, objs = [], []
    for s in SOURCES:
        obj = os.path.join(objdir, os.path.basename(s) + ".o")
        objs.append(obj)
        src = os.path.join(CSRC, s)
        if incremental and os.path.exists(obj) and all(os.path.getmtime(d) < os.path.getmtime(obj) for d in [src] + hdrs):
            continue
        cmd = [nvcc] + NVCC_FLAGS + extra + ["-c", "-o", obj, src]
        procs.append((obj, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for obj, pr in procs:
        out = pr.communicate()[0]
        if verbose or pr.returncode:
            sys.stderr.write(out)
        failed |= pr.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed building " + out_path)
    r = subprocess.run([nvcc, "-shared", "-o", out_path] + objs + ["-lz"], capture_output=True, text=True)      # zlib: the BGZF container of b200_bcfio.c
    if verbose or r.returncode:
        sys.stderr.write(r.stdout + r.stderr)
    if r.returncode:
        raise RuntimeError("nvcc failed linking " + out_path)
    return out_path


def build_variant(out_path, defines, verbose=False):
    """Experimental builds with extra -D flags (scripts/ use this for register-cap sweeps)."""
    return _compile_link(out_path, ["-D" + d for d in defines], verbose)


def build(force=False, verbose=False):
    if not force and not _stale():
        return LIB
    os.makedirs(os.path.dirname(LIB), exist_ok=True)
    return _compile_link(LIB, ["-Xptxas", "-v"] if verbose else [], verbose, incremental=not force and not verbose)


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))     # no flag: incremental rebuild of what is stale
