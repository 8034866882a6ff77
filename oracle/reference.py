"""Optional install of the unmodified original package (lucidrains/naturalspeech2-pytorch) into oracle/_ref/.

bench.py's CPU legs (`--impl reference`, the in-run parity check, the aligner and prompt-encoder CPU timings) run
the original code when it is installed here, and the torch port of the oracle otherwise.  Nothing else needs it:
the tests compare with fixtures recorded from it under tests/golden/.  `build()` installs it when NS2_REFERENCE_SRC
names a checkout of the original project: a pure-Python install with no dependencies and no package index (the
third-party modules it imports but the benchmarked path never touches are stubbed by bench.import_reference).
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
import tempfile
from pathlib import Path

REF_DIR = Path(__file__).resolve().parent / "_ref"


def installed() -> bool:
    return (REF_DIR / "naturalspeech2_pytorch").exists()


def install(src: str | None = None) -> None:
    """pip-install the checkout at `src` (default: $NS2_REFERENCE_SRC; nothing to do when unset) into REF_DIR."""
    src = src or os.environ.get("NS2_REFERENCE_SRC")
    if not src or installed():
        return
    with tempfile.TemporaryDirectory() as tmp:
        copy = Path(tmp) / "reference"
        shutil.copytree(src, copy)          # setuptools writes build files next to the sources
        cmd = [sys.executable, "-m", "pip", "install", "--no-index", "--no-build-isolation", "--no-deps",
               "--target", str(REF_DIR), str(copy)]
        res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        print(f"reference install into {REF_DIR} failed (bench.py's CPU legs will use the oracle port):\n"
              f"{res.stderr[-400:]}")
    else:
        print(f"installed the reference into {REF_DIR}")
