"""Installs the original project's Modin (unmodified) into ``oracle/_ref/`` (git-ignored).

Modin is pure Python, so installing it means copying its ``modin`` package tree.  The copy is what the plug-in
tests, ``tools/dist_check.py --api modin`` and ``bench.py`` (its default front door and its ``--impl reference`` arm)
import as real ``modin.pandas``.  The source tree is ``$MODIN_REFERENCE_SRC``, or ``DEFAULT_SRC`` if that is not
set.  Where the source cannot be read, an existing ``oracle/_ref`` is kept as it is (built elsewhere and shipped
with the tree), and without one the tests that need Modin skip.
"""

from __future__ import annotations

import os
import shutil

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.path.join(HERE, "_ref")
DEFAULT_SRC = "/root/reference"


def source() -> str:
    return os.environ.get("MODIN_REFERENCE_SRC") or DEFAULT_SRC


def installed() -> bool:
    return os.path.isfile(os.path.join(REF, "modin", "__init__.py"))


def build() -> str | None:
    """Copies ``<source>/modin`` to ``oracle/_ref/modin``.  Returns the installed path, or None when no source was
    readable and nothing was installed before."""
    src = os.path.join(source(), "modin")
    if not os.access(os.path.join(src, "__init__.py"), os.R_OK):
        return os.path.join(REF, "modin") if installed() else None
    os.makedirs(REF, exist_ok=True)
    tmp = os.path.join(REF, ".modin.tmp")
    shutil.rmtree(tmp, ignore_errors=True)
    shutil.copytree(src, tmp, ignore=shutil.ignore_patterns("__pycache__", "*.pyc"))
    dst = os.path.join(REF, "modin")
    shutil.rmtree(dst, ignore_errors=True)
    os.rename(tmp, dst)
    return dst


if __name__ == "__main__":
    print(build())
