"""Recipe for oracle/_ref: compile the UNMODIFIED reference package for the CPU reference arm.

    python oracle/build_ref.py        # needs /root/reference (this container); writes oracle/_ref/gigaam_ref.zip + MANIFEST.json

The reference is a Python package whose hot path is torch CPU ops.  Its modules are byte-compiled from the sources
where they lie under /root/reference (py_compile, nothing is copied as source and nothing of it enters the repository:
oracle/_ref/ is git-ignored) into one import archive, oracle/_ref/gigaam_ref.zip, which -- like the built .so -- travels to
the GPU box with the snapshot; /root/reference does not exist there.  `oracle/ref_loader.py` imports the package from the
archive with the three absent third-party modules (hydra, omegaconf, soundfile) stubbed, the same way oracle/make_golden.py
imports it from /root/reference.  Test infrastructure only: nothing under gigaam_b200/ imports it; `bench.py --impl
reference` times it (cpu_baseline.kind = "reference") and tests/test_oracle_golden.py pins the oracle port against it.
"""
from __future__ import annotations

import hashlib
import json
import os
import py_compile
import subprocess
import sys
import tempfile
import zipfile
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
REF = Path(os.environ.get("GIGAAM_REFERENCE", "/root/reference"))
OUT = ROOT / "oracle" / "_ref"
ARCHIVE = OUT / "gigaam_ref.zip"


def build_ref(quiet: bool = False):
    src = REF / "gigaam"
    try:
        present = src.is_dir()
    except OSError:          # not readable by this user: the same as absent
        present = False
    if not present:
        if not quiet:
            print(f"{src} not present: keeping whatever oracle/_ref already holds")
        return ARCHIVE if ARCHIVE.is_file() else None
    OUT.mkdir(parents=True, exist_ok=True)
    manifest = {}
    with tempfile.TemporaryDirectory() as tmp, zipfile.ZipFile(ARCHIVE, "w", zipfile.ZIP_DEFLATED) as z:
        for f in sorted(src.glob("*.py")):
            pyc = Path(tmp) / (f.stem + ".pyc")
            # hash-based, unchecked: valid without the source file next to it and independent of timestamps
            py_compile.compile(str(f), cfile=str(pyc), dfile=f"gigaam/{f.name}", doraise=True,
                               invalidation_mode=py_compile.PycInvalidationMode.UNCHECKED_HASH)
            z.write(pyc, f"gigaam/{f.stem}.pyc")
            manifest[f.name] = hashlib.sha256(f.read_bytes()).hexdigest()
    head = subprocess.run(["git", "-C", str(REF), "rev-parse", "HEAD"], capture_output=True, text=True).stdout.strip()
    (OUT / "MANIFEST.json").write_text(json.dumps({"source": str(src), "commit": head, "python": sys.version.split()[0],
                                                   "sha256_of_sources": manifest}, indent=1))
    if not quiet:
        print(f"compiled {len(manifest)} reference modules into {ARCHIVE}")
    return ARCHIVE


if __name__ == "__main__":
    sys.exit(0 if build_ref() else 1)
