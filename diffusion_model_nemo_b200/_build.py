"""In-tree build of libdmn_b200.so (nvcc, sm_100a only).  Used by __graft_entry__.build() and `python -m diffusion_model_nemo_b200._build`."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libdmn_b200.so")
SOURCES = ["plan.cu", "kernels_simt.cu", "conv_tcgen05.cu", "linattn_mma.cu", "attn_fused.cu", "sampler.cu", "api_layers.cu", "ode.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xptxas", "-v",
    "-Xcompiler", "-fPIC,-O2,-Wall,-Wno-unused-function", "--expt-relaxed-constexpr",
]


def needs_rebuild() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".h"))]
    deps += [os.path.join(HERE, "..", "include", "dmn_b200.h"), os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build_variant(path: str, extra_flags) -> str:
    """Build a differently-configured copy of the library (e.g. -DDMN_TC_TRACE_BUILD=1 for tools/trace_conv.py) at `path`;
    select it with DMN_LIB_PATH.  Objects go to a scratch directory, the in-tree build is untouched."""
    import tempfile

    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    with tempfile.TemporaryDirectory() as tmp:
        procs, objs = [], []
        for src in SOURCES:
            obj = os.path.join(tmp, src.replace(".cu", ".o"))
            objs.append(obj)
            cmd = [nvcc, *[f for f in NVCC_FLAGS if f not in ("-Xptxas", "-v")], *extra_flags, "-c", os.path.join(CSRC, src), "-o", obj]
            procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        for src, p in procs:
            out, _ = p.communicate()
            if p.returncode != 0:
                sys.stderr.write(out)
                raise RuntimeError(f"nvcc failed on {src}")
        out = subprocess.run([nvcc, "-shared", "-o", path, *objs, "-lcudart"], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        if out.returncode != 0:
            sys.stderr.write(out.stdout)
            raise RuntimeError("link failed")
    return path


def build(force: bool = False, verbose: bool = False) -> str:
    """Concurrent callers (several ranks / pytest workers on a stale tree) serialise on a file lock; objects and the library are
    written to a scratch directory and the .so is moved into place atomically, so nobody ever dlopens a half-linked file."""
    import fcntl
    import tempfile

    if not force and not needs_rebuild():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    with open(os.path.join(HERE, ".build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        if not force and not needs_rebuild():      # another process built it while we waited
            return LIB
        with tempfile.TemporaryDirectory(dir=HERE, prefix=".build_") as tmp:
            objs, procs = [], []
            for src in SOURCES:
                obj = os.path.join(tmp, src.replace(".cu", ".o"))
                objs.append(obj)
                cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
                procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
            log = []
            failed = None
            for src, p in procs:
                out, _ = p.communicate()
                log.append(f"==== {src}\n{out}")
                if p.returncode != 0 and failed is None:
                    failed = src
            if failed:
                sys.stderr.write("\n".join(log))
                raise RuntimeError(f"nvcc failed on {failed}")
            tmp_lib = os.path.join(tmp, "libdmn_b200.so")
            out = subprocess.run([nvcc, "-shared", "-o", tmp_lib, *objs, "-lcudart"], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
            if out.returncode != 0:
                sys.stderr.write(out.stdout)
                raise RuntimeError("link failed")
            os.replace(tmp_lib, LIB)
        with open(os.path.join(CSRC, "build.log"), "w") as f:
            f.write("\n".join(log))
        if verbose:
            print("\n".join(log))
    return LIB


if __name__ == "__main__":
    if "--variant" in sys.argv:       # python -m diffusion_model_nemo_b200._build --variant tools/libdmn_x.so -DDMN_TC_TRACE_BUILD=1 ...
        i = sys.argv.index("--variant")
        print(build_variant(sys.argv[i + 1], sys.argv[i + 2:]))
    else:
        print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
