"""Compile-when-stale builder of the oracle's C restatements (test infrastructure).

Every library is built with gcc and -ffp-contract=off: no product is fused into an add, as in
x86-64 builds of R.  It goes next to its source, or -- when the tree is read-only -- into a
per-user temporary directory.
"""
import os
import subprocess
import tempfile

_HERE = os.path.dirname(os.path.abspath(__file__))
# /usr/bin/gcc is named explicitly when present, as in oracle/Makefile
_GCC = "/usr/bin/gcc" if os.access("/usr/bin/gcc", os.X_OK) else "gcc"


def _compile(src, out, openmp):
    base = [_GCC, "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-Wall", "-Wextra", "-o", out, src]
    if openmp and subprocess.call(base[:1] + ["-fopenmp"] + base[1:]) == 0:
        return
    subprocess.check_call(base)


def build_shared(name, openmp=False, force=False):
    """oracle/<name>.c -> liboracle_<stem>.so (stem: name without "_oracle"), compiled when missing
    or older than the source; openmp=True adds -fopenmp where gcc supports it.  Returns its path."""
    src = os.path.join(_HERE, name + ".c")
    so = os.path.join(_HERE, "liboracle_%s.so" % name.replace("_oracle", ""))
    if not force and os.path.exists(so) and os.path.getmtime(so) >= os.path.getmtime(src):
        return so
    if os.access(_HERE, os.W_OK):
        _compile(src, so, openmp)
        return so
    out = os.path.join(tempfile.gettempdir(), "recoup_b200_%s_%d.so" % (os.path.basename(so)[3:-3], os.getuid()))
    if force or not os.path.exists(out) or os.path.getmtime(out) < os.path.getmtime(src):
        _compile(src, out, openmp)
    return out
