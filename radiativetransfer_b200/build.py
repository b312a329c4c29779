"""Builds librtb200.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels with the repo snapshot)."""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "librtb200.so")
SOURCES = ["api.cu", "diffuse_uniform.cu", "diffuse_amr.cu", "point_source.cu", "chemistry.cu", "multi.cu", "scattering.cu", "ng.cu", "dust.cu", "octree_build.cu", "geometry.cpp", "point_host.cpp", "uvb_host.cpp"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "--use_fast_math=false", "-Xcompiler", "-fPIC,-O2,-ffp-contract=off,-fno-fast-math", "-Xptxas", "-v",
]


def _nvcc():
    return shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"


def needs_build():
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "rtb200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return OUT
    bdir = os.path.join(HERE, "build")
    os.makedirs(bdir, exist_ok=True)
    flags = [f for f in NVCC_FLAGS if f != "--use_fast_math=false"]

    def compile_one(src):
        path = os.path.join(CSRC, src)
        obj = os.path.join(bdir, src.rsplit(".", 1)[0] + ".o")
        r = subprocess.run([_nvcc()] + flags + ["-x", "cu", "-c", path, "-o", obj], capture_output=True, text=True)
        return src, obj, r

    from concurrent.futures import ThreadPoolExecutor
    sources = [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    with ThreadPoolExecutor(max_workers=min(len(sources), os.cpu_count() or 1)) as ex:   # one nvcc per translation unit
        results = list(ex.map(compile_one, sources))
    objs = []
    for src, obj, r in results:
        if verbose or r.returncode:
            sys.stderr.write(r.stdout + r.stderr)
        if r.returncode:
            raise RuntimeError(f"nvcc failed on {src}")
        with open(obj + ".ptxas.txt", "w") as f:
            f.write(r.stderr)
        objs.append(obj)
    cmd = [_nvcc(), "-shared", "-o", OUT] + objs + ["-lcudart", "-ldl", "-lpthread"]
    subprocess.check_call(cmd)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
