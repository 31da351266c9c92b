"""Recipe for ``oracle/_ref``: the UNMODIFIED reference (openai/gym 0.26.2), copied from its source tree.

Test / measurement infrastructure, not product code.  The reference is pure Python, so installing it is a plain copy
of its ``gym`` package into ``oracle/_ref/gym`` (git-ignored; no pip, no network).  Nothing is copied into the
repository's history, and nothing under ``gym_b200/`` imports it.

    python oracle/make_ref.py            # (re)build oracle/_ref when the reference's source tree is readable

Consumers (``tests/``, ``bench.py``'s ``cpu_baseline_python`` leg) go through ``oracle.ref_gym.import_reference()``.
"""
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
REFERENCE = "/root/reference"
TARGET = os.path.join(HERE, "_ref")


def build(force=False):
    """Returns the path of the installed reference, or None when its source tree cannot be read here."""
    marker = os.path.join(TARGET, "gym", "version.py")
    if os.path.exists(marker) and not force:
        return TARGET
    src = os.path.join(REFERENCE, "gym")
    if not os.path.isfile(os.path.join(src, "version.py")):
        return TARGET if os.path.exists(marker) else None
    # copy beside the installed package and rename, so that an interrupted copy never looks installed
    staging = os.path.join(TARGET, "gym.partial")
    shutil.rmtree(staging, ignore_errors=True)
    os.makedirs(TARGET, exist_ok=True)
    shutil.copytree(src, staging, ignore=shutil.ignore_patterns("__pycache__"))
    for root, dirs, files in os.walk(staging):   # the source tree is read-only; the copy must stay removable
        for d in dirs:
            os.chmod(os.path.join(root, d), 0o755)
        for f in files:
            os.chmod(os.path.join(root, f), 0o644)
    os.chmod(staging, 0o755)
    shutil.rmtree(os.path.join(TARGET, "gym"), ignore_errors=True)
    os.rename(staging, os.path.join(TARGET, "gym"))
    return TARGET


if __name__ == "__main__":
    path = build(force=True)
    print(path or f"the reference's source tree ({REFERENCE}) is not readable here", file=sys.stdout if path else sys.stderr)
    sys.exit(0 if path else 1)
