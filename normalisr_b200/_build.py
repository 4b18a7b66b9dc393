"""Build the CUDA library in-tree: normalisr_b200/libnsr_b200.so (sm_100a only)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libnsr_b200.so")
SOURCES = ["api.cu", "basis.cu", "binnet.cu", "de4.cu", "grouped.cu", "lcpm.cu", "normvar.cu", "sympinv.cu", "textio.cu", "hostcopy.cu", "residual.cu", "contract_simt.cu", "contract_umma.cu", "contract_umma_splitk.cu"]
HEADERS = ["nsr_common.cuh", "epilogue.cuh", "pvalue.cuh", "contract_route.h", os.path.join("..", "..", "include", "normalisr_b200.h")]
INCLUDES = {"contract_umma_splitk.cu": ["contract_umma.cu"]}      # sources that #include another source


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def _compile_one(args):
    src, obj, verbose, env = args
    cmd = [_nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
           "-Xcompiler", "-fPIC", "-Xptxas", "-v" if verbose else "-warn-spills", "-c", "-o", obj, src]
    res = subprocess.run(cmd, capture_output=True, text=True, env=env)
    return src, res.returncode, res.stdout + res.stderr


def build(force=False, verbose=False):
    """One object per source (compiled in parallel, recompiled only when the source or a header is newer),
    then one link: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo ... -shared."""
    if not force and not stale():
        return LIB
    from concurrent.futures import ThreadPoolExecutor
    env = dict(os.environ)
    env.pop("CC", None)
    env.pop("CXX", None)
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    hdr_t = max(os.path.getmtime(os.path.join(CSRC, h)) for h in HEADERS)
    hdr_t = max(hdr_t, os.path.getmtime(os.path.abspath(__file__)))
    jobs, objs = [], []
    for sname in SOURCES:
        src = os.path.join(CSRC, sname)
        obj = os.path.join(objdir, sname[:-3] + ".o")
        objs.append(obj)
        src_t = max([os.path.getmtime(src)] + [os.path.getmtime(os.path.join(CSRC, d)) for d in INCLUDES.get(sname, ())])
        if force or verbose or not os.path.exists(obj) or os.path.getmtime(obj) < max(hdr_t, src_t):
            jobs.append((src, obj, verbose, env))
    with ThreadPoolExecutor(max_workers=min(8, max(1, len(jobs)))) as ex:
        results = list(ex.map(_compile_one, jobs))
    for src, rc, out in results:
        if verbose or rc != 0:
            sys.stderr.write(out)
        if rc != 0:
            raise RuntimeError("nvcc failed on %s:\n%s" % (src, out[-4000:]))
    res = subprocess.run([_nvcc(), "-shared", "-o", LIB] + objs, capture_output=True, text=True, env=env)
    if res.returncode != 0:
        raise RuntimeError("nvcc link failed:\n" + res.stderr[-4000:])
    return LIB


if __name__ == "__main__":
    print(build(force="-f" in sys.argv, verbose="-v" in sys.argv))
