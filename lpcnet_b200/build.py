"""Builds liblpcnet_b200.so (sm_100a) in-tree with nvcc.  No torch, no JIT cache: the .so travels with the repo
snapshot to the GPU box.  `python -m lpcnet_b200.build` or `lpcnet_b200.build.build()`."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
SO = os.path.join(HERE, "liblpcnet_b200.so")
HOST_SOURCES = ["model.cu", "frame_kernels.cu", "batch_api.cu", "lpcnet_api.cu", "microbench.cu", "multi_api.cu", "blob_io.cu", "enc_kernels.cu"]
KERNEL_SOURCES = ["sample_kernel.cu", "sample_kernel_f32.cu", "sample_kernel_f32n.cu"]   # compiled once per GRU_A size (-DLPCNET_NA=<na>, engine.h)
NA_SIZES = [128, 256, 384]
HOST_SOURCES = [f for f in HOST_SOURCES if os.path.exists(os.path.join(CSRC, f))]


def units():
    """(source file, object name, extra -D flags) of every translation unit."""
    u = [(s, s.replace(".cu", ".o"), []) for s in HOST_SOURCES]
    for na in NA_SIZES:
        u += [(s, s.replace(".cu", "_na%d.o" % na), ["-DLPCNET_NA=%d" % na]) for s in KERNEL_SOURCES]
    return u


def _compile_all(objdir, extra_defs, log):
    """nvcc every unit (in parallel: the nine kernel units dominate the build time)."""
    from concurrent.futures import ThreadPoolExecutor
    os.makedirs(objdir, exist_ok=True)

    def one(u):
        src, obj, defs = u
        o = os.path.join(objdir, obj)
        cmd = [NVCC] + FLAGS + defs + ["-D%s" % d for d in extra_defs] + ["-c", os.path.join(CSRC, src), "-o", o]
        r = subprocess.run(cmd, capture_output=True, text=True)
        return u, o, r
    objs = []
    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:
        for u, o, r in ex.map(one, units()):
            log.append("==== %s %s\n%s" % (u[0], " ".join(u[2]), r.stderr))
            if r.returncode != 0:
                sys.stderr.write(r.stdout + r.stderr)
                raise RuntimeError("nvcc failed on %s %s" % (u[0], u[2]))
            objs.append(o)
    return objs
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
         "-fmad=false",                    # never contract a*b+c: the pinned oracle build uses -ffp-contract=off
         "-Xcompiler", "-fPIC,-fvisibility=hidden,-ffp-contract=off", "-Xptxas", "-v"]


def needs_build():
    if not os.path.exists(SO):
        return True
    t = os.path.getmtime(SO)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", f) for f in ("lpcnet.h", "lpcnet_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build_variant(name, defines):
    """Tuning aid: build lpcnet_b200/variants/lib_<name>.so with extra -D flags (e.g. LPCNET_TRACE=1)."""
    vdir = os.path.join(HERE, "variants")
    log = []
    os.makedirs(vdir, exist_ok=True)
    objs = _compile_all(os.path.join("/tmp", "lpcnet_b200_variant_obj_" + name), defines, log)     # objects outside the tree: the gpurun snapshot stays small
    for blk in log:
        if blk.startswith("==== sample_kernel.cu -DLPCNET_NA=384"):
            print(name, [l.strip() for l in blk.splitlines() if "registers" in l or "spill" in l][-2:])
    so = os.path.join(vdir, "lib_%s.so" % name)
    subprocess.check_call([NVCC, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", so] + objs + ["-lcudart"])
    return so


def build(force=False, verbose=False):
    if not force and not needs_build():
        return SO
    log = []
    objs = _compile_all(os.path.join(HERE, "_obj"), [], log)
    r = subprocess.run([NVCC, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", SO] + objs + ["-lcudart"],
                       capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("link failed")
    with open(os.path.join(HERE, "_obj", "ptxas.log"), "w") as f:
        f.write("\n".join(log))
    if verbose:
        print("\n".join(log))
    return SO


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
