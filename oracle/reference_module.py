"""Load the UNMODIFIED reference package (davitpapikyan/Normalizing-Flow-with-Diffusion-Prior-Model) as a comparator.

TEST INFRASTRUCTURE ONLY: used by ``bench.py --impl reference`` / ``--impl reference-gpu`` (the reference arms), by
``tests/test_dropin_overlay.py`` and by the golden-vector generators — never by the product path.

The reference is not part of this repository: point ``NFDPM_REFERENCE`` at a checkout of it to enable the comparisons
(without it they are skipped).  It is pure Python on PyTorch, so "building" it is packing its source tree:
``stage()`` (called by ``__graft_entry__.build()``) writes ONE archive, ``baseline/_ref/reference_src.tar.gz`` —
git-ignored, so no reference source enters the history or sits in the tree as files, but it travels with a copy of the
working tree to a machine without the checkout.  ``find()`` unpacks it into the system's temporary
directory (once per archive content) and ``import_reference()`` imports ``normalizing_flow`` from there with the reference's
non-hot-path dependencies that this image lacks (aim, skimage, cleanfid, ignite: logging / data / metrics code, reference
normalizing_flow/utils.py:4, trainer.py:8-13, data/utils.py:9, metrics/compute.py:21-30) stubbed by MagicMock.

The reference package has the same import name as the product's drop-in mirror; a process imports ONE of them
(``bench.py`` runs the reference arms in their own processes).
"""
from __future__ import annotations

import hashlib
import os
import shutil
import sys
import tarfile
import tempfile
from unittest.mock import MagicMock

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STAGED = os.path.join(ROOT, "baseline", "_ref")
SOURCE = os.environ.get("NFDPM_REFERENCE") or None
STUBS = ["aim", "skimage", "skimage.transform", "cleanfid", "cleanfid.fid", "cleanfid.features", "cleanfid.utils",
         "cleanfid.resize", "ignite", "ignite.metrics"]


ARCHIVE = os.path.join(STAGED, "reference_src.tar.gz")
_SKIP = ("media", ".git", "__pycache__")


def stage(src: str = SOURCE, dst: str = STAGED) -> bool:
    """Pack the reference's Python tree (no media, no VCS data) into ``dst``/reference_src.tar.gz.  Returns False when
    ``src`` is unset or absent."""
    if not src or not os.path.isdir(os.path.join(src, "normalizing_flow")):
        return False
    if os.path.isdir(dst):
        shutil.rmtree(dst)
    os.makedirs(dst)

    def keep(ti: tarfile.TarInfo):
        parts = ti.name.split("/")
        if any(p in _SKIP for p in parts) or ti.name.endswith((".pyc", ".png", ".gif", ".jpg")):
            return None
        ti.mtime, ti.uid, ti.gid, ti.uname, ti.gname = 0, 0, 0, "", ""       # reproducible archive -> stable unpack directory
        return ti
    with tarfile.open(os.path.join(dst, "reference_src.tar.gz"), "w:gz") as tf:
        tf.add(src, arcname="reference", filter=keep)
    return True


def find() -> str | None:
    """Directory holding an importable copy of the reference tree: the staged archive unpacked under the temporary directory,
    else the checkout NFDPM_REFERENCE names."""
    if os.path.isfile(ARCHIVE):
        h = hashlib.sha1(open(ARCHIVE, "rb").read()).hexdigest()[:12]
        out = os.path.join(tempfile.gettempdir(), f"nfdpm_reference_{h}")
        root = os.path.join(out, "reference")
        if not os.path.isdir(os.path.join(root, "normalizing_flow")):
            tmp = out + f".{os.getpid()}"
            with tarfile.open(ARCHIVE, "r:gz") as tf:
                tf.extractall(tmp, filter="data")
            try:
                os.rename(tmp, out)
            except OSError:                    # another process unpacked it meanwhile
                shutil.rmtree(tmp, ignore_errors=True)
        return root
    if SOURCE and os.path.isdir(os.path.join(SOURCE, "normalizing_flow")):
        return SOURCE
    return None


def import_reference(path: str | None = None):
    """-> the reference's ``normalizing_flow`` module (raises ImportError when no copy is available or when another
    package of that name — the product's mirror — is already imported in this process)."""
    path = path or find()
    if path is None:
        raise ImportError("no copy of the reference: neither baseline/_ref/reference_src.tar.gz (staged by "
                          f"__graft_entry__.build()) nor NFDPM_REFERENCE={SOURCE!r} exists")
    have = sys.modules.get("normalizing_flow")
    if have is not None:
        if os.path.realpath(getattr(have, "__file__", "")).startswith(os.path.realpath(path)):
            return have
        raise ImportError("a different 'normalizing_flow' package is already imported in this process")
    for m in STUBS:
        sys.modules.setdefault(m, MagicMock())
    sys.path.insert(0, path)
    import normalizing_flow as nf  # noqa: E402
    assert os.path.realpath(nf.__file__).startswith(os.path.realpath(path)), nf.__file__
    return nf
