"""Recipe: compile the REFERENCE's own Cython MISE (code/src/libmise/mise.pyx — the only native source in the reference,
SURVEY §2.2) from a reference source tree into oracle/_ref/ (git-ignored, never copied into the repo's history).  Nothing in
the build or the test suite needs it: tools/bench_aux.py times it where it exists, and its `mise.MISE` has the interface of
oracle/mise_oracle.MISE, so it can stand in for the oracle in tests/test_cpu_mise.py to re-pin the oracle round by round.
usage: python oracle/build_ref_mise.py <reference>/code/src/libmise/mise.pyx"""
import os
import subprocess
import sys
import sysconfig

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "_ref")


def build(src):
    os.makedirs(OUT, exist_ok=True)
    ext = sysconfig.get_config_var("EXT_SUFFIX")
    so = os.path.join(OUT, "mise" + ext)
    if os.path.exists(so) and os.path.getmtime(so) >= os.path.getmtime(src):
        return so
    cpp = os.path.join(OUT, "mise.cpp")
    subprocess.run([sys.executable, "-m", "cython", "--cplus", "-3", src, "-o", cpp], check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    import numpy as np

    inc = [sysconfig.get_paths()["include"], np.get_include()]
    cmd = ["g++", "-O2", "-shared", "-fPIC", "-std=c++14", "-w"] + [f"-I{i}" for i in inc] + ["-o", so, cpp]
    subprocess.run(cmd, check=True)
    os.remove(cpp)
    return so


if __name__ == "__main__":
    print(build(sys.argv[1]))
