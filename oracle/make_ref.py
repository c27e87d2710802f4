#!/usr/bin/env python
"""Install the UNMODIFIED reference into oracle/_ref (git-ignored; optional: bench.py times the oracle
port instead when it is absent): `pip install --no-index --no-build-isolation --no-deps --target oracle/_ref <copy>`.

TEST / BENCH INFRASTRUCTURE.  The install is made from a writable scratch copy in the temporary
directory because the reference source may be read-only and setuptools writes egg-info/build
directories into the source tree.
`--no-deps`: gymnasium / treevalue / jsonargparse / ... are not installable offline; the stand-ins
under oracle/refstubs replace them at run time (oracle/run_reference.py).  Recorded outcome:
DESIGN.md §6.  No reference source file is copied into the tracked tree.
"""
import os
import shutil
import stat
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
REF_SRC = "/root/reference"
TARGET = os.path.join(HERE, "_ref")


def installed():
    return os.path.isfile(os.path.join(TARGET, "openrl", "__init__.py"))


def _make_writable(tree):
    """copytree keeps the source's mode bits; a read-only source would give a copy setuptools cannot build in."""
    for d, _, files in os.walk(tree):
        for p in [d] + [os.path.join(d, f) for f in files if not os.path.islink(os.path.join(d, f))]:
            os.chmod(p, os.stat(p).st_mode | stat.S_IWUSR)


def main(force=False):
    if installed() and not force:
        print("oracle/_ref already holds the reference install")
        return True
    if not os.path.isdir(REF_SRC):
        print("reference source absent: using the existing oracle/_ref" if installed() else "reference source absent: no oracle/_ref")
        return installed()
    tmp = tempfile.mkdtemp(prefix="openrl_ref_")
    try:
        src = os.path.join(tmp, "reference")
        shutil.copytree(REF_SRC, src, ignore=shutil.ignore_patterns(".git"))
        _make_writable(src)
        if os.path.isdir(TARGET):
            shutil.rmtree(TARGET)
        cmd = [sys.executable, "-m", "pip", "install", "--no-index", "--no-build-isolation", "--no-deps", "--no-cache-dir",
               "--target", TARGET, src]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            print(r.stdout[-2000:], r.stderr[-2000:])
            return False
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    print("installed the reference into", TARGET)
    return installed()


if __name__ == "__main__":
    sys.exit(0 if main(force="--force" in sys.argv) else 1)
