"""Compiles the upstream PaSCo package (`pasco/` of an upstream checkout) into sourceless bytecode under oracle/_ref/, for
the drop-in tests (tests/test_dropin_reference.py), which run the unmodified upstream model on the engine.

    python oracle/build_ref.py

The checkout is PASCO_REFERENCE, or DEFAULT_CHECKOUT when that is unset.  Without a checkout nothing changes, so a
compiled package made earlier stays in place.  oracle/_ref/ holds no source text and is not committed; the bytecode
belongs to the Python version that compiled it."""
import os
import py_compile
import shutil
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DST = os.path.join(ROOT, "oracle", "_ref")
DEFAULT_CHECKOUT = "/root/reference"


def build_ref(src=None) -> bool:
    """Returns True when oracle/_ref/pasco was (re)compiled from a checkout."""
    src = src or os.environ.get("PASCO_REFERENCE") or DEFAULT_CHECKOUT
    pkg = os.path.join(src, "pasco")
    if not os.path.isdir(pkg):
        return False
    out = os.path.join(DST, "pasco")
    tmp = out + ".tmp"
    shutil.rmtree(tmp, ignore_errors=True)
    for dirpath, dirnames, files in os.walk(pkg):
        dirnames[:] = [d for d in dirnames if d != "__pycache__"]
        rel = os.path.relpath(dirpath, pkg)
        for f in files:
            if f.endswith(".py"):
                # legacy location (next to where the .py would be): the import system loads it without a source file
                dst = os.path.join(tmp, rel, f[:-3] + ".pyc")
                py_compile.compile(os.path.join(dirpath, f), cfile=dst, dfile=os.path.join("pasco", rel, f), doraise=True,
                                   invalidation_mode=py_compile.PycInvalidationMode.UNCHECKED_HASH)
    shutil.rmtree(out, ignore_errors=True)
    os.replace(tmp, out)
    return True


if __name__ == "__main__":
    print("compiled" if build_ref(sys.argv[1] if len(sys.argv) > 1 else None) else "no upstream checkout found")
