"""Installs the unmodified LibKGE package (`kge`) from its source tree into oracle/_ref (git-ignored).

The kge_b200 plugin subclasses LibKGE's own model and job classes, and the tests and bench.py compare the plugin's
jobs against LibKGE's own jobs, so both need `kge` importable.  LibKGE is pure Python: installing it is copying its
modules and the yaml files it loads at run time (the package data its setup.py leaves out), nothing else.  The
result is self-contained, so it can be carried to a machine that has no LibKGE source tree.  Nothing of LibKGE enters
the repository.

    python oracle/install_ref.py [SOURCE_TREE]      (default: $KGE_REFERENCE_SRC, else /root/reference)
"""
from __future__ import annotations

import os
import shutil
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
TARGET = os.path.join(HERE, "_ref")
DEFAULT_SOURCE = "/root/reference"


def source_tree() -> str | None:
    """The LibKGE source tree to install from, or None if there is none (or it cannot be read)."""
    src = os.environ.get("KGE_REFERENCE_SRC", DEFAULT_SOURCE)
    return src if os.access(os.path.join(src, "kge", "model"), os.R_OK | os.X_OK) else None


def installed() -> bool:
    return os.path.isdir(os.path.join(TARGET, "kge", "model"))


def install(src: str) -> str:
    """Copies every .py / .yaml file of src/kge into oracle/_ref/kge; returns oracle/_ref."""
    files = []
    for d, _, names in os.walk(os.path.join(src, "kge")):
        files += [os.path.relpath(os.path.join(d, f), src) for f in names if f.endswith((".py", ".yaml"))]
    if not any(f.endswith(os.path.join("kge", "model", "__init__.py")) for f in files):
        raise RuntimeError(f"no LibKGE package under {src}")
    # build beside the target and swap it in, so an interrupted install never leaves a partial tree behind
    tmp = tempfile.mkdtemp(prefix="_ref.", dir=HERE)
    try:
        os.chmod(tmp, 0o755)
        for f in files:
            os.makedirs(os.path.join(tmp, os.path.dirname(f)), exist_ok=True)
            shutil.copyfile(os.path.join(src, f), os.path.join(tmp, f))
        shutil.rmtree(TARGET, ignore_errors=True)
        os.rename(tmp, TARGET)
    except BaseException:
        shutil.rmtree(tmp, ignore_errors=True)
        raise
    return TARGET


if __name__ == "__main__":
    src = sys.argv[1] if len(sys.argv) > 1 else source_tree()
    if src is None:
        sys.exit("LibKGE source tree not found: pass it as an argument or set KGE_REFERENCE_SRC")
    print(install(src))
