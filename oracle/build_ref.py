"""Build the reference's own Version C hot path (Cython + OpenMP) into oracle/_ref/.

TEST / BASELINE INFRASTRUCTURE ONLY -- nothing in the product package imports this.

What it does (SURVEY.md section 8c recipe, BASELINE.md section 3 step 1):
  * reads the reference tree where it lies (the argument, else CRB_REFERENCE_SRC; read-only),
  * mirrors the `crender` package (+ the `objects/` assets the README flow needs) into the git-ignored
    build directory oracle/_ref/ -- a build output, never committed,
  * applies the two BUILD-ONLY changes the reference needs to compile with gcc:
      - `# distutils: extra_{compile,link}_args = /openmp`  ->  `-fopenmp`
        (crender/cy/pixel_buffer_filler/advanced_pixel_buffer_filler.pyx:2-3 hard-codes the MSVC flag),
      - Cython directive legacy_implicit_noexcept=True (the Cython-0.29 semantics the author measured with;
        stock Cython 3 takes the GIL after every candidate pixel, SURVEY.md section 6),
  * compiles with /usr/bin/gcc, default -O2, no -march=native / -ffast-math (would change f32 bits).
No arithmetic is touched.  Import the result with  sys.path.insert(0, "oracle/_ref").
"""
import os
import re
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
DST = os.path.join(HERE, "_ref")

_SETUP = r'''
from setuptools import setup
from Cython.Build import cythonize
import numpy
setup(
    name="crender_ref_oracle", version="0.0.1",
    ext_modules=cythonize(
        ["crender/cy/pixel_buffer_filler/advanced_pixel_buffer_filler.pyx",
         "crender/cy/pixel_buffer_filler/math_utils.pyx"],
        compiler_directives={"legacy_implicit_noexcept": True, "language_level": "3"},
        quiet=True),
    include_dirs=[numpy.get_include()],
)
'''


def built(dst=DST):
    d = os.path.join(dst, "crender", "cy", "pixel_buffer_filler")
    if not os.path.isdir(d):
        return False
    names = os.listdir(d)
    return (any(n.startswith("advanced_pixel_buffer_filler.") and n.endswith(".so") for n in names)
            and any(n.startswith("math_utils.") and n.endswith(".so") for n in names))


def build(src=None, dst=DST, force=False):
    """src: a checkout of the reference (default: the CRB_REFERENCE_SRC environment variable)."""
    if built(dst) and not force:
        return dst
    src = src or os.environ.get("CRB_REFERENCE_SRC")
    if not src or not os.path.isdir(os.path.join(src, "crender")):
        raise FileNotFoundError(f"no reference checkout at {src!r} (pass its path or set CRB_REFERENCE_SRC)")
    if os.path.isdir(dst):
        shutil.rmtree(dst)
    os.makedirs(dst)
    shutil.copytree(os.path.join(src, "crender"), os.path.join(dst, "crender"))
    shutil.copytree(os.path.join(src, "objects"), os.path.join(dst, "objects"))
    os.makedirs(os.path.join(dst, "output"), exist_ok=True)
    for root, _, files in os.walk(dst):          # the mirror of a read-only tree is read-only too
        os.chmod(root, 0o755)
        for f in files:
            os.chmod(os.path.join(root, f), 0o644)
    pyx = os.path.join(dst, "crender/cy/pixel_buffer_filler/advanced_pixel_buffer_filler.pyx")
    with open(pyx) as f:
        text = f.read()
    text, n = re.subn(r"(# distutils: extra_(?:compile|link)_args = )/openmp", r"\1-fopenmp", text)
    assert n == 2, "expected exactly two /openmp build lines"
    with open(pyx, "w") as f:
        f.write(text)
    with open(os.path.join(dst, "_build_oracle.py"), "w") as f:
        f.write(_SETUP)
    env = dict(os.environ, CC="/usr/bin/gcc", LDSHARED="/usr/bin/gcc -shared")
    env.pop("CFLAGS", None)
    subprocess.check_call([sys.executable, "_build_oracle.py", "build_ext", "--inplace", "-q"],
                          cwd=dst, env=env)
    shutil.rmtree(os.path.join(dst, "build"), ignore_errors=True)
    assert built(dst)
    return dst


if __name__ == "__main__":
    paths = [a for a in sys.argv[1:] if a != "--force"]      # usage: build_ref.py [REFERENCE_CHECKOUT] [--force]
    print(build(paths[0] if paths else None, force="--force" in sys.argv))
