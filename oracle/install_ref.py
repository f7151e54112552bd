"""Install the UNMODIFIED reference (underdoc-wang/MPGCN) into `oracle/_ref/` (git-ignored).

The reference is six flat Python modules with no setup.py / pyproject.toml, so pip cannot install it (recorded in DESIGN.md);
"installing" it is copying its files to `oracle/_ref/` and putting that directory on sys.path, exactly how its own Main.py
finds its siblings.  Nothing under oracle/_ref is tracked or edited; bench.py's reference arms and the trainer drop-in tests
import it from there, and fall back (bench.py: the torch port) or skip (tests) where it is absent.

The reference checkout is read from $MPGCN_REFERENCE_DIR, by default from the same place oracle/gen_golden.py reads it:

    MPGCN_REFERENCE_DIR=/path/to/MPGCN python oracle/install_ref.py
"""
import os
import shutil
import sys

SRC = os.environ.get("MPGCN_REFERENCE_DIR", "/root/reference")
DST = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")


def main() -> int:
    if not os.path.isdir(SRC):
        print(f"reference not found at {SRC}: keeping whatever is in {DST}")
        return 0
    os.makedirs(DST, exist_ok=True)
    n = 0
    for f in sorted(os.listdir(SRC)):
        if f.endswith(".py") or f in ("LICENSE", "README.md"):
            shutil.copyfile(os.path.join(SRC, f), os.path.join(DST, f))
            n += 1
    print(f"copied {n} files from {SRC} to {DST}")
    return 0


if __name__ == "__main__":
    sys.exit(main())
