"""Build the runnable copy of the reference (TEST INFRASTRUCTURE ONLY).

Two outputs:

* ``oracle/_ref/_c_llr*.so`` -- the reference's only native component
  (``/root/reference/adapted/detect/_c_llr.pyx``) cythonized and compiled from the source
  where it lies.  The build product is git-ignored but travels to the GPU box, where it serves
  as the "reference" arm for the LLR-gains kernel.
* ``oracle/_ref/pkg`` (git-ignored like everything under ``oracle/_ref``, so it never enters the
  history, but it travels to the GPU box with the snapshot): the runnable copy of the python
  reference package with the two py>=3.11 dataclass fixes applied, the compiled ``_c_llr`` next to
  its pyx, plus a ``bottleneck`` stand-in that forwards to :mod:`oracle.bn_restate`.
  ``oracle/make_golden.py`` and the oracle-vs-reference tests import it from there, and
  ``bench.py --impl reference`` times it as the CPU arm (``cpu_baseline.kind = "reference"``): the
  reference's own ``combined_detect_cnn`` / ``combined_detect_llr2`` under a process pool.  Nothing
  under ``tests -m gpu`` or ``smoke()`` touches it.

No reference source is committed to the repository.
"""
from __future__ import annotations

import os
import re
import shutil
import subprocess
import sys
import sysconfig

REFERENCE = "/root/reference"
HERE = os.path.dirname(os.path.abspath(__file__))
REF_OUT = os.path.join(HERE, "_ref")
SCRATCH = os.environ.get("ADB_REF_SCRATCH", "/tmp/adapted_ref_scratch")


def reference_present() -> bool:
    return os.path.isfile(os.path.join(REFERENCE, "adapted", "detect", "_c_llr.pyx"))


def _ext_suffix() -> str:
    return sysconfig.get_config_var("EXT_SUFFIX")


def ref_so_path() -> str:
    return os.path.join(REF_OUT, "_c_llr" + _ext_suffix())


def build_c_llr(force: bool = False) -> str:
    """cythonize + g++ the reference pyx (no -march => no FMA contraction, like a stock build)."""
    import numpy as np

    out = ref_so_path()
    src = os.path.join(REFERENCE, "adapted", "detect", "_c_llr.pyx")
    if os.path.exists(out) and not force and os.path.getmtime(out) >= os.path.getmtime(src):
        return out
    os.makedirs(REF_OUT, exist_ok=True)
    tmp = os.path.join(SCRATCH, "_build")
    os.makedirs(tmp, exist_ok=True)
    cpp = os.path.join(tmp, "_c_llr.cpp")
    subprocess.check_call(
        [sys.executable, "-m", "cython", "-3", "--cplus", "-o", cpp, src],
        stdout=subprocess.DEVNULL,
        stderr=subprocess.DEVNULL,
    )
    inc = [np.get_include(), sysconfig.get_paths()["include"]]
    cmd = ["g++", "-O2", "-fPIC", "-shared", "-w", "-DNPY_NO_DEPRECATED_API=NPY_1_7_API_VERSION"]
    cmd += ["-I" + i for i in inc] + [cpp, "-o", out]
    subprocess.check_call(cmd)
    return out


_FIELD_RE = re.compile(r"^(\s+)(\w+): (\w+) = (\w+Config)\(\)$", re.M)


PKG = os.path.join(REF_OUT, "pkg")


def package_present() -> bool:
    return os.path.exists(os.path.join(PKG, "built.stamp"))


def build_scratch_package(force: bool = False) -> str:
    """Patched python copy of the reference in oracle/_ref/pkg; returns the directory to put on sys.path."""
    root = PKG
    os.makedirs(REF_OUT, exist_ok=True)
    stamp = os.path.join(root, "built.stamp")
    if os.path.exists(stamp) and not force:
        return root
    if os.path.exists(root):
        shutil.rmtree(root)
    os.makedirs(root)
    shutil.copytree(os.path.join(REFERENCE, "adapted"), os.path.join(root, "adapted"))
    for rel in ("adapted/config/sig_proc.py", "adapted/config/config.py"):
        p = os.path.join(root, rel)
        s = open(p).read()
        s = _FIELD_RE.sub(r"\1\2: \3 = field(default_factory=\4)", s)
        s = s.replace("from dataclasses import dataclass\n", "from dataclasses import dataclass, field\n", 1)
        open(p, "w").write(s)
    so = build_c_llr(force)
    shutil.copy(so, os.path.join(root, "adapted", "detect", os.path.basename(so)))
    bn = os.path.join(root, "bottleneck")
    os.makedirs(bn)
    with open(os.path.join(bn, "__init__.py"), "w") as f:
        f.write(
            "import os, sys\n"
            "sys.path.insert(0, os.path.abspath(os.path.join(os.path.dirname(__file__), '..', '..', '..', '..')))\n"
            "from oracle.bn_restate import move_mean, move_var\n"
            "__version__ = '1.3.7'\n"
        )
    open(stamp, "w").write("ok\n")
    return root


def kernel_available() -> bool:
    """the reference's compiled _c_llr can be loaded: from its source, or prebuilt in oracle/_ref"""
    return reference_present() or os.path.exists(ref_so_path())


def load_c_llr():
    """the reference's compiled _c_llr module (built first where the source is present)"""
    import importlib.util

    so = build_c_llr() if reference_present() else ref_so_path()
    spec = importlib.util.spec_from_file_location("_c_llr", so)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def import_reference():
    """Put the runnable copy on sys.path and return the reference's ``adapted`` package (built first where
    /root/reference exists; on the GPU box the prebuilt oracle/_ref/pkg is used as it is)."""
    root = build_scratch_package() if reference_present() else PKG
    if not package_present():
        raise ImportError("oracle/_ref/pkg has not been built (python -m oracle.build_ref where /root/reference exists)")
    if root not in sys.path:
        sys.path.insert(0, root)
    import warnings

    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        import adapted  # noqa: F401
        import adapted.detect.combined  # noqa: F401
    return sys.modules["adapted"]


if __name__ == "__main__":
    if not reference_present():
        print("reference not present; nothing to build")
        sys.exit(0)
    print(build_c_llr(force="--force" in sys.argv))
    print(build_scratch_package(force="--force" in sys.argv))
