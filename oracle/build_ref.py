"""TEST INFRASTRUCTURE ONLY -- build ``oracle/_ref``: the REFERENCE itself (pysteps v1.21.3 under
/root/reference) in compiled form, so that it can travel to the GPU box (which has no
/root/reference) and run there as the checker and as the CPU arm of bench.py.

    python oracle/build_ref.py            (also run by __graft_entry__.build() when the reference is present)

What it writes, all under oracle/_ref/ (git-ignored, not gpurun-ignored), all built from the
sources where they lie -- no source file is copied:
  pysteps/**/*.pyc            every module of the package compiled to bytecode (sourceless import;
                              the package's tests/ and scripts/ are left out)
  pysteps/motion/_vet.*.so    the reference's two Cython extensions, cythonized in a scratch
  pysteps/motion/_proesmans.*.so  directory and compiled with the flags of setup.py:27-28
                              (-fopenmp -O3 -ffast-math)
``import pysteps`` itself needs jsmin / matplotlib (absent in this image); the modules are
imported under a stub namespace package (oracle/refimport.py), which runs each submodule's own
code unchanged.
"""
import importlib.util
import os
import py_compile
import shutil
import subprocess
import sys
import sysconfig
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.environ.get("PYSTEPS_REFERENCE", "/root/reference")
OUT = os.path.join(HERE, "_ref")
SKIP_DIRS = {"tests", "scripts", "__pycache__"}


def available():
    return os.path.isdir(os.path.join(REF, "pysteps"))


def _stale(dst, src):
    return (not os.path.exists(dst)) or os.path.getmtime(src) > os.path.getmtime(dst)


def compile_modules():
    n = 0
    root = os.path.join(REF, "pysteps")
    for dirpath, dirnames, filenames in os.walk(root):
        dirnames[:] = [d for d in dirnames if d not in SKIP_DIRS]
        rel = os.path.relpath(dirpath, REF)
        for fn in filenames:
            src = os.path.join(dirpath, fn)
            if fn.endswith(".py"):
                dst = os.path.join(OUT, rel, fn + "c")
                if _stale(dst, src):
                    os.makedirs(os.path.dirname(dst), exist_ok=True)
                    py_compile.compile(src, cfile=dst, dfile=os.path.join("pysteps-reference", rel, fn), doraise=True)
                n += 1
    return n


def build_extension(name):
    """pysteps/motion/<name>.pyx -> oracle/_ref/pysteps/motion/<name>.<abi>.so"""
    import numpy
    src = os.path.join(REF, "pysteps", "motion", name + ".pyx")
    suffix = sysconfig.get_config_var("EXT_SUFFIX")
    dst = os.path.join(OUT, "pysteps", "motion", name + suffix)
    if not _stale(dst, src):
        return dst
    os.makedirs(os.path.dirname(dst), exist_ok=True)
    with tempfile.TemporaryDirectory() as tmp:
        c_file = os.path.join(tmp, name + ".c")
        subprocess.check_call([sys.executable, "-m", "cython", "-3", src, "-o", c_file])
        cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
        inc = [sysconfig.get_paths()["include"], numpy.get_include()]
        so = os.path.join(tmp, name + suffix)
        subprocess.check_call([cc, "-shared", "-fPIC", "-fopenmp", "-O3", "-ffast-math", "-w"]
                              + [f"-I{i}" for i in inc] + [c_file, "-o", so])
        shutil.copyfile(so, dst)
    return dst


def build():
    if not available():
        return False
    n = compile_modules()
    if importlib.util.find_spec("Cython") is None:
        # the bytecode alone serves the pure-Python modules; vet / proesmans of the reference and
        # the tests that run its nowcast loop then skip
        print("oracle/build_ref.py: Cython is not installed; the reference's _vet / _proesmans extensions "
              "are not built")
    else:
        for ext in ("_vet", "_proesmans"):
            build_extension(ext)
    with open(os.path.join(OUT, "README"), "w") as f:
        f.write("Built by oracle/build_ref.py from /root/reference (pysteps v1.21.3): bytecode of the package "
                f"({n} modules) and its two Cython extensions.  Test infrastructure; not product code.\n")
    return True


if __name__ == "__main__":
    ok = build()
    print("oracle/_ref built" if ok else "reference not present; nothing built")
