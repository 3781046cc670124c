"""Recipe for oracle/_ref/ - the UNMODIFIED reference class, staged so it can run on the GPU box too
(ORACLE / TEST INFRASTRUCTURE ONLY; never imported by the product).

The reference's path is one Python file, /root/reference/swarmdb/" main.py" (the name starts with a space).
Where /root/reference exists (the build container) this recipe copies that file byte for byte into
oracle/_ref/swarmdb_reference_main.py and writes its sha256 beside it.  oracle/_ref/ is git-ignored (reference
sources never enter the history) but NOT gpurun-ignored, so the copy travels with the snapshot and
`bench.py`'s reference-python leg can time the reference's own code on the GPU box's host cores.
`oracle/ref_loader.py` loads it - through the same two documented shims - when /root/reference is absent.

    python -m oracle.build_ref        (also run by __graft_entry__.build())
"""
from __future__ import annotations

import hashlib
import shutil
import sys

from oracle.ref_loader import REFERENCE_MAIN as SOURCE, STAGED_MAIN as STAGED, readable_file

REF_DIR = STAGED.parent


def build(quiet: bool = False) -> bool:
    """Returns True when oracle/_ref holds the reference file (freshly staged or already there)."""
    if not readable_file(SOURCE):
        if not quiet:
            print(f"oracle/_ref: {SOURCE} not present here; keeping whatever is staged", file=sys.stderr)
        return STAGED.is_file()
    REF_DIR.mkdir(exist_ok=True)
    shutil.copyfile(SOURCE, STAGED)
    digest = hashlib.sha256(STAGED.read_bytes()).hexdigest()
    (REF_DIR / "SHA256").write_text(f"{digest}  swarmdb/ main.py (staged unmodified from /root/reference)\n")
    if not quiet:
        print(f"oracle/_ref: staged {SOURCE} ({STAGED.stat().st_size} bytes, sha256 {digest[:16]}...)")
    return True


if __name__ == "__main__":
    sys.exit(0 if build() else 1)
