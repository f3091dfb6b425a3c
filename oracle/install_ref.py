"""Stage the UNMODIFIED reference for bench.py's reference arm and the tests:  python oracle/install_ref.py

joliGEN is a plain Python source tree (no setup.py / pyproject.toml), so there is nothing to compile: the staged form
is a copy of the Python packages its training step imports, under oracle/_ref/.  That directory is git-ignored
(reference sources never enter the history) and travels with the built tree to machines that have no reference
checkout.  __graft_entry__.build() runs it whenever the reference checkout (JG_REFERENCE_ROOT) is readable.
"""
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
DEST = os.path.join(HERE, "_ref")
SRC = os.environ.get("JG_REFERENCE_ROOT", "/root/reference")
PACKAGES = ["models", "options", "util", "data"]
FILES = ["train.py", "LICENSE"]
EXAMPLES = ["example_ddpm_mario.json", "example_gan_horse2zebra.json", "example_ddpm_unetref_viton.json",
            "example_ddpm_vid_mario.json", "example_b2b_vid_mario.json"]


def install(force=False):
    if not os.path.isdir(SRC):
        return None
    stamp = os.path.join(DEST, ".installed")
    if os.path.exists(stamp) and not force:
        return DEST
    shutil.rmtree(DEST, ignore_errors=True)
    os.makedirs(DEST)
    ignore = shutil.ignore_patterns("__pycache__", "*.pyc", "*.so")   # (op/ loads its .cpp / .cu at import)
    for pkg in PACKAGES:
        shutil.copytree(os.path.join(SRC, pkg), os.path.join(DEST, pkg), ignore=ignore)
    for f in FILES:
        if os.path.exists(os.path.join(SRC, f)):
            shutil.copy2(os.path.join(SRC, f), os.path.join(DEST, f))
    os.makedirs(os.path.join(DEST, "examples"))
    for f in EXAMPLES:
        p = os.path.join(SRC, "examples", f)
        if os.path.exists(p):
            shutil.copy2(p, os.path.join(DEST, "examples", f))
    with open(stamp, "w") as f:
        f.write("copied from %s\n" % SRC)
    return DEST


if __name__ == "__main__":
    print(install(force="--force" in sys.argv))
