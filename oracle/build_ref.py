"""Build recipe for oracle/_ref/: the reference YOLACT tree (Python) compiled to sourceless bytecode, so that tests can
run the reference's own modules (tests/test_eval_drop_in.py imports its eval.py unchanged) from a build product of
this repository instead of a tree outside it.  oracle/_ref/ is git-ignored.

The reference is taken from YOLACT_REFERENCE, else from DEFAULT_REFERENCE.  Without a readable one nothing is built
and the tests that need it skip."""
import os
import py_compile
import shutil
import warnings

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "_ref", "yolact")
DEFAULT_REFERENCE = "/root/reference"   # where the upstream checkout is looked for when YOLACT_REFERENCE is unset


def reference_root():
    root = os.environ.get("YOLACT_REFERENCE") or DEFAULT_REFERENCE
    return root if os.path.isfile(os.path.join(root, "eval.py")) and os.access(root, os.R_OK | os.X_OK) else None


def build():
    """Compiles every .py of the reference to OUT/<same path>.pyc (importable without the source); returns OUT, or None
    when there is no reference.  Files that do not compile on this Python cannot be imported either and are left out."""
    root = reference_root()
    if root is None:
        return None
    tmp = OUT + ".tmp"
    shutil.rmtree(tmp, ignore_errors=True)
    for d, dirs, files in os.walk(root):
        dirs[:] = sorted(x for x in dirs if not x.startswith("."))
        for f in sorted(files):
            if f.endswith(".py"):
                rel = os.path.relpath(os.path.join(d, f), root)
                try:
                    with warnings.catch_warnings():   # the reference's own SyntaxWarnings (invalid escapes)
                        warnings.simplefilter("ignore")
                        py_compile.compile(os.path.join(d, f), cfile=os.path.join(tmp, rel + "c"), dfile=rel,
                                           doraise=True)
                except py_compile.PyCompileError:
                    pass
    shutil.rmtree(OUT, ignore_errors=True)
    os.replace(tmp, OUT)
    return OUT


if __name__ == "__main__":
    print("built", build())
