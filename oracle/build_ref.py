"""TEST / MEASUREMENT INFRASTRUCTURE ONLY -- never imported by the product (sample_factory_b200/).

Installs the UNMODIFIED reference (sample-factory 2.1.3) into oracle/_ref (git-ignored) for the reference arm of bench.py
(oracle/ref_driver.py) and for tests/test_boundary.py, which runs the reference's own sf_examples scripts against this
repository.  The source is a checkout of the reference at $SFB200_REFERENCE_SRC (default /root/reference); without one
nothing is installed and those two fall back (the oracle port) or skip.

`pip install --no-deps`: the reference's third-party dependencies (gymnasium, signal-slot-mp, faster-fifo, tensorboardX,
colorlog) are not needed to install it, and oracle/ref_shims.py stands in for them at import time.
"""
from __future__ import annotations

import os
import shutil
import stat
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_DIR = os.path.join(ROOT, "oracle", "_ref")


def installed(ref_dir: str = REF_DIR) -> bool:
    return os.path.isfile(os.path.join(ref_dir, "sample_factory", "algo", "learning", "learner.py"))


def install(src: str | None = None, ref_dir: str = REF_DIR) -> bool:
    """Install the reference into `ref_dir` unless it is there already.  Returns whether it is installed afterwards."""
    src = src or os.environ.get("SFB200_REFERENCE_SRC", "/root/reference")
    if installed(ref_dir):
        return True
    if not os.path.isfile(os.path.join(src, "setup.py")):
        return False
    with tempfile.TemporaryDirectory() as tmp:
        # setuptools writes build/ next to setup.py: work on a copy, made writable (the checkout may be read-only and
        # copytree keeps its modes)
        work = os.path.join(tmp, "ref_src")
        shutil.copytree(src, work, symlinks=True)
        os.chmod(work, os.stat(work).st_mode | stat.S_IWUSR)
        for d, dirs, files in os.walk(work):
            for name in dirs + files:
                p = os.path.join(d, name)
                if not os.path.islink(p):
                    os.chmod(p, os.stat(p).st_mode | stat.S_IWUSR)
        res = subprocess.run([sys.executable, "-m", "pip", "install", "--no-index", "--no-build-isolation", "--no-deps",
                              "--no-cache-dir", "--target", ref_dir, work], capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(f"installing the reference into {ref_dir} failed (the bench falls back to the oracle port):\n"
                         + res.stdout[-1500:] + res.stderr[-1500:] + "\n")
        shutil.rmtree(ref_dir, ignore_errors=True)
    return installed(ref_dir)
