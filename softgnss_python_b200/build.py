"""Compile the CUDA sources in csrc/ into the in-tree shared library (sm_100a only).

    python -m softgnss_python_b200.build

``-fmad=false``: float64 loop-filter / code-phase arithmetic must round every operation
separately, as numpy does (SURVEY.md appendix A.2); hot float32 loops call fmaf() explicitly.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libsoftgnss_b200.so")
SOURCES = ["sgx_api.cu", "sgx_track.cu", "sgx_synth.cu", "sgx_acq.cu", "sgx_pfa.cu", "sgx_fine.cu", "sgx_bitsync.cu", "sgx_nav.cu", "sgx_quality.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-fmad=false", "-Xcompiler", "-fPIC", "-Xptxas", "-v", "--use_fast_math=false"]


def _sources():
    return [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = _sources() + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cuh")]
    deps.append(os.path.join(os.path.dirname(HERE), "include", "softgnss_b200.h"))
    return any(os.path.getmtime(d) > t for d in deps)


def force_all():
    return os.environ.get("SGX_BUILD_ALL", "") == "1"


def build_native(force=False, verbose=False):
    """nvcc -> in-tree libsoftgnss_b200.so; the translation units are compiled in parallel."""
    if not force and not needs_build():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    flags = [f for f in NVCC_FLAGS if f != "--use_fast_math=false"]
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    procs = []
    hdrs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    hdrs.append(os.path.join(os.path.dirname(HERE), "include", "softgnss_b200.h"))
    hdr_time = max(os.path.getmtime(h) for h in hdrs)
    objs_cached = []
    for src in _sources():
        obj = os.path.join(objdir, os.path.basename(src)[:-3] + ".o")
        log = obj + ".log"
        # per-object cache (sgx_acq.cu alone takes minutes): rebuild when the source or any header is newer
        if (not force_all() and os.path.exists(obj) and os.path.exists(log)
                and os.path.getmtime(obj) > max(os.path.getmtime(src), hdr_time)):
            objs_cached.append((obj, open(log).read()))
            continue
        procs.append((src, obj, subprocess.Popen([nvcc] + flags + ["-c", "-o", obj, src], stdout=subprocess.PIPE,
                                                 stderr=subprocess.PIPE, text=True)))
    report, objs = [c[1] for c in objs_cached], [c[0] for c in objs_cached]
    for src, obj, p in procs:
        out, err = p.communicate()
        report.append(err)
        if p.returncode == 0:
            with open(obj + ".log", "w") as f:
                f.write(err)
        if verbose or p.returncode != 0:
            sys.stderr.write(out + err)
        if p.returncode != 0:
            raise RuntimeError("nvcc failed on " + src)
        objs.append(obj)
    res = subprocess.run([nvcc, "-shared", "-o", LIB] + objs, capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("link failed")
    with open(os.path.join(HERE, "csrc", "ptxas_report.txt"), "w") as f:
        f.write("".join(report))
    return LIB


if __name__ == "__main__":
    print(build_native(force=True, verbose="-v" in sys.argv))
