"""TEST INFRASTRUCTURE ONLY -- builds oracle/_ref/fiber, the reference pool package (uber/fiber @ ad6faf02)
compiled to sourceless bytecode, which ``bench.py``'s CPU arm (``cpu_baseline``, ``--impl reference``)
imports to time the reference itself.

Only bytecode is written: no source file of the reference enters this tree.  One constant is changed
before compiling, ``socket_lib = "nanomsg"`` -> ``"zmq"`` in ``fiber/socket.py``, because nnpy (the
nanomsg binding) is not installable offline while pyzmq is; results are ``func(arg)`` placed by index,
so the transport does not change them (tests/golden/make_golden.py makes the same change).

    python -m oracle.ref_pyc            # or: __graft_entry__.build()

The reference checkout is read from ``$FIBER_REFERENCE`` (default ``/root/reference``).  Where it is
absent, an ``oracle/_ref/fiber`` built earlier is left as it is.  The bytecode is specific to the
Python minor version that compiled it.
"""
import importlib.util
import marshal
import os
import shutil

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "_ref")
REFERENCE = os.environ.get("FIBER_REFERENCE", "/root/reference")
PATCH = ("fiber/socket.py", 'socket_lib = "nanomsg"', 'socket_lib = "zmq"')


def _pyc(code):
    """A .pyc image that the sourceless loader accepts: magic, flags 0 (timestamp form, never checked
    without a source file next to it), mtime 0, size 0, marshalled code."""
    return importlib.util.MAGIC_NUMBER + bytes(12) + marshal.dumps(code)


def build():
    """-> True when oracle/_ref/fiber exists afterwards."""
    src_pkg = os.path.join(REFERENCE, "fiber")
    dst_pkg = os.path.join(OUT, "fiber")
    if not os.path.isdir(src_pkg):
        return os.path.isdir(dst_pkg)
    tmp = dst_pkg + ".tmp"
    shutil.rmtree(tmp, ignore_errors=True)
    patched = False
    for dirpath, dirnames, filenames in os.walk(src_pkg):
        dirnames[:] = sorted(d for d in dirnames if d != "__pycache__")
        for name in sorted(f for f in filenames if f.endswith(".py")):
            rel = os.path.relpath(os.path.join(dirpath, name), REFERENCE).replace(os.sep, "/")
            with open(os.path.join(dirpath, name), encoding="utf-8") as fh:
                text = fh.read()
            if rel == PATCH[0]:
                assert text.count(PATCH[1]) == 1, "%s: expected one %r" % (rel, PATCH[1])
                text, patched = text.replace(PATCH[1], PATCH[2]), True
            code = compile(text, rel, "exec", dont_inherit=True)
            out = os.path.join(tmp, os.path.relpath(dirpath, src_pkg), name[:-3] + ".pyc")
            os.makedirs(os.path.dirname(out), exist_ok=True)
            with open(out, "wb") as fh:
                fh.write(_pyc(code))
    assert patched, "%s not found under %s" % (PATCH[0], REFERENCE)
    shutil.rmtree(dst_pkg, ignore_errors=True)
    os.replace(tmp, dst_pkg)
    return True


if __name__ == "__main__":
    print(build())
