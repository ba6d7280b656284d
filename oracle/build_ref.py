#!/usr/bin/env python
"""ORACLE TOOLING (test infrastructure, NOT product code): build the REAL reference for the tests that run its classes.

Byte-compiles every module of the LightX2V package (`$LIGHTX2V_REFERENCE/lightx2v`, default `/root/reference/lightx2v`, the
reference checkout's usual location) into sourceless `.pyc` files under the git-ignored `oracle/_ref/lightx2v`, where
`oracle/ref_loader.py` imports it.  Nothing of the reference enters the history, and the build output needs no checkout at run time.
`__graft_entry__.build()` runs this; where no checkout exists it is a no-op and the tests that need the package skip.

    python oracle/build_ref.py
"""
import os
import py_compile
import shutil
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.environ.get("LIGHTX2V_REFERENCE", "/root/reference")
DST = os.path.join(ROOT, "oracle", "_ref")


def build() -> bool:
    src_pkg = os.path.join(SRC, "lightx2v")
    if not os.path.isdir(src_pkg):
        return False
    dst_pkg = os.path.join(DST, "lightx2v")
    if os.path.isdir(dst_pkg):
        shutil.rmtree(dst_pkg)
    for dirpath, dirnames, filenames in os.walk(src_pkg):
        dirnames[:] = [d for d in dirnames if d != "__pycache__"]
        rel = os.path.relpath(dirpath, SRC)
        for name in filenames:
            if name.endswith(".py"):
                # a module.pyc with no module.py beside it is imported directly (sourceless import)
                py_compile.compile(os.path.join(dirpath, name), cfile=os.path.join(DST, rel, name + "c"), dfile=os.path.join(rel, name),
                                   doraise=True)
    return True


if __name__ == "__main__":
    ok = build()
    print("built" if ok else f"{SRC} holds no LightX2V package: nothing to do", DST)
    sys.exit(0)
