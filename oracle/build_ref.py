"""Recipe for ``oracle/_ref``: the UNMODIFIED reference modules of the hot path, placed where they can travel.

TEST / BASELINE INFRASTRUCTURE ONLY.  The reference is four pure-Python files (modules.py, models.py, sampling.py,
utils.py: no build system, no native code), so "building" it is copying those files, byte for byte, from the read-only
checkout at /root/reference into ``oracle/_ref/``.  That directory is git-ignored (reference sources never enter the
history) but NOT gpurun-ignored, so it reaches the GPU box like the repo's own built ``.so``.

Consumers (and only these): ``bench.py --impl reference`` / the ``cpu_baseline`` leg time the reference's own
``DiffusionProcess`` on the host cores (``kind: "reference"``), and the ``eager_gpu`` leg runs the same modules on the
B200 through cuDNN / cuBLAS (the bar the hand-written path has to beat).  When ``oracle/_ref`` is absent those legs fall
back to the oracle port (``kind: "port"``).  The product path never touches either.

    python oracle/build_ref.py            # copies if /root/reference exists, reports otherwise
"""
from __future__ import annotations

import hashlib
import shutil
import sys
from pathlib import Path

REF = Path("/root/reference")
DST = Path(__file__).resolve().parent / "_ref"
FILES = ("modules.py", "models.py", "sampling.py", "utils.py")


def _present(d: Path) -> bool:
    """True when `d` holds the four reference files.  A directory this user may not read counts as absent."""
    try:
        return all((d / f).exists() for f in FILES)
    except OSError:
        return False


def build(verbose: bool = True) -> bool:
    """Returns True when oracle/_ref holds the four reference files (freshly copied or already there)."""
    if not _present(REF):
        ok = _present(DST)
        if verbose:
            print(f"[build_ref] {REF} not present; oracle/_ref {'already populated' if ok else 'unavailable'}")
        return ok
    DST.mkdir(exist_ok=True)
    for f in FILES:
        shutil.copyfile(REF / f, DST / f)
    digest = hashlib.sha256(b"".join((DST / f).read_bytes() for f in FILES)).hexdigest()[:16]
    (DST / "SOURCE.txt").write_text(f"copied verbatim from {REF} ({', '.join(FILES)}); sha256[:16] = {digest}\n")
    if verbose:
        print(f"[build_ref] oracle/_ref <- {REF} ({digest})")
    return True


if __name__ == "__main__":
    sys.exit(0 if build() else 1)
