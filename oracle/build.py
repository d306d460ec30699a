"""Build recipe for the oracle's native pieces.  TEST INFRASTRUCTURE ONLY.

* ``build_oracle_c()``  gcc -> ``oracle/liboracle_c.so`` from ``oracle/oracle_c.c``
  (our own C restatement; travels to the GPU box as a built .so).
* ``build_ref()``       compiles the REFERENCE's own Cython module
  ``/root/reference/pgl/graph_kernel.pyx`` together with its vendored METIS 5.1.0
  (``/root/reference/pgl/third_party/metis``) from the sources where they lie, outputs
  only into ``oracle/_ref/`` (git-ignored, not gpurun-ignored).  Mirrors the source/include
  lists of ``/root/reference/setup.py:82-117`` without running the reference's build
  system.  No reference source is copied into the repository; the generated
  ``graph_kernel.cpp`` is an intermediate inside ``oracle/_ref/build``.  The METIS objects
  are also linked alone into ``oracle/_ref/libmetis_i64.so``.

``load_ref_graph_kernel()`` imports the built module directly (bypassing
``pgl/__init__.py:21`` which needs paddle) and returns None when it has not been built
(e.g. on the GPU box before the snapshot's .so is there).
"""
import glob
import importlib.util
import os
import subprocess
import sys
import sysconfig

HERE = os.path.dirname(os.path.abspath(__file__))
REF = "/root/reference"
REF_OUT = os.path.join(HERE, "_ref")


def _run(cmd, **kw):
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, **kw)
    if r.returncode != 0:
        raise RuntimeError("command failed: %s\n%s" % (" ".join(cmd), r.stdout[-4000:]))
    return r.stdout


def _newer(target, sources):
    if not os.path.exists(target):
        return False
    t = os.path.getmtime(target)
    return all(os.path.getmtime(s) <= t for s in sources)


def oracle_c_path():
    return os.path.join(HERE, "liboracle_c.so")


def build_oracle_c(force=False, out=None):
    """An up-to-date oracle/liboracle_c.so is reused; otherwise gcc writes the library to `out`
    (default: oracle/liboracle_c.so)."""
    src = os.path.join(HERE, "oracle_c.c")
    if not force and _newer(oracle_c_path(), [src]):
        return oracle_c_path()
    out = out or oracle_c_path()
    _run(["gcc", "-O3", "-march=native", "-fopenmp", "-fPIC", "-shared", "-std=c11",
          "-o", out, src])
    return out


def ref_so_path():
    suffix = sysconfig.get_config_var("EXT_SUFFIX") or ".so"
    return os.path.join(REF_OUT, "graph_kernel" + suffix)


def ref_metis_path():
    return os.path.join(REF_OUT, "libmetis_i64.so")


def build_ref(force=False, jobs=8):
    """Compile the reference's graph_kernel.pyx + METIS into oracle/_ref/, and link the METIS objects
    alone into oracle/_ref/libmetis_i64.so (what pgl_b200/build.py:build_metis makes from the same
    sources with the same flags) for the METIS tests where the package's own copy cannot be built."""
    pyx = os.path.join(REF, "pgl", "graph_kernel.pyx")
    out = ref_so_path()
    if not os.path.exists(pyx):
        return out if os.path.exists(out) else None
    if not force and os.path.exists(out) and os.path.exists(ref_metis_path()):
        return out
    import numpy

    bdir = os.path.join(REF_OUT, "build")
    os.makedirs(bdir, exist_ok=True)
    metis = os.path.join(REF, "pgl", "third_party", "metis")
    incs = ["-I" + os.path.join(metis, "include"), "-I" + os.path.join(metis, "GKlib"),
            "-I" + os.path.join(metis, "libmetis"), "-I" + os.path.join(REF, "pgl"),
            "-I" + numpy.get_include(), "-I" + sysconfig.get_paths()["include"]]
    cpp = os.path.join(bdir, "graph_kernel.cpp")
    _run([sys.executable, "-m", "cython", "--cplus", "-3", pyx, "-o", cpp])
    csrcs = (glob.glob(os.path.join(metis, "GKlib", "*.c"))
             + glob.glob(os.path.join(metis, "*.c"))
             + glob.glob(os.path.join(metis, "libmetis", "*.c")))
    objs = []
    procs = []
    # the reference builds every file with g++ (language="c++", setup.py:111); the METIS
    # C files are valid C, compile them as C with gcc to stay warning-tolerant.
    for s in csrcs:
        o = os.path.join(bdir, os.path.basename(os.path.dirname(s)) + "_" +
                         os.path.basename(s)[:-2] + ".o")
        objs.append(o)
        if os.path.exists(o) and not force:
            continue
        procs.append((s, subprocess.Popen(
            ["gcc", "-O2", "-fPIC", "-w", "-c", s, "-o", o] + incs,
            stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        if len(procs) >= jobs:
            s0, p0 = procs.pop(0)
            o0, _ = p0.communicate()
            if p0.returncode != 0:
                raise RuntimeError("gcc failed on %s\n%s" % (s0, o0[-3000:]))
    for s0, p0 in procs:
        o0, _ = p0.communicate()
        if p0.returncode != 0:
            raise RuntimeError("gcc failed on %s\n%s" % (s0, o0[-3000:]))
    o_main = os.path.join(bdir, "graph_kernel.o")
    _run(["g++", "-O2", "-fPIC", "-w", "-std=c++11", "-c", cpp, "-o", o_main] + incs)
    _run(["g++", "-shared", "-o", out, o_main] + objs + ["-lm"])
    metis_objs = [o for o in objs if os.path.basename(o).startswith(("GKlib_", "libmetis_"))]
    _run(["gcc", "-shared", "-o", ref_metis_path()] + metis_objs + ["-lm"])
    return out


def load_ref_graph_kernel():
    p = ref_so_path()
    if not os.path.exists(p):
        return None
    spec = importlib.util.spec_from_file_location("graph_kernel", p)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


if __name__ == "__main__":
    print(build_oracle_c(force="--force" in sys.argv))
    print(build_ref(force="--force" in sys.argv))
