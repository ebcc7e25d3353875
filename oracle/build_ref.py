"""Install the unmodified reference package (google/TensorNetwork 0.4.6) into `oracle/_ref/`.

`python -m oracle.build_ref [SOURCE]`; `__graft_entry__.build()` runs it.  SOURCE is a checkout of the reference
(the directory holding `tensornetwork/`), by default `$TN_REFERENCE_SRC`, else `/root/reference`.  The package is
pure Python, so installing it is a copy of its `tensornetwork/` tree; nothing in it is changed.  `oracle/_ref/` is a
build product (git-ignored).  The tests that drive the reference's own callers on the project's backends, and the
reference arm of bench.py, import it from there through baseline/refenv.py.  Without a readable source the install is
skipped and those users see no reference.
"""
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
DEST = os.path.join(HERE, "_ref")


def default_source():
  return os.environ.get("TN_REFERENCE_SRC", "/root/reference")


def installed():
  return os.path.isfile(os.path.join(DEST, "tensornetwork", "__init__.py"))


def build(source=None):
  """Copies SOURCE/tensornetwork to oracle/_ref/tensornetwork unless it is already there.  Returns True when the
  reference is installed afterwards."""
  if installed():
    return True
  pkg = os.path.join(source or default_source(), "tensornetwork")
  if not os.access(os.path.join(pkg, "__init__.py"), os.R_OK):
    return False
  tmp = DEST + ".tmp"
  shutil.rmtree(tmp, ignore_errors=True)
  shutil.copytree(pkg, os.path.join(tmp, "tensornetwork"),
                  ignore=shutil.ignore_patterns("__pycache__", "*.pyc"))
  for root, dirs, files in os.walk(tmp):          # the source tree is read-only; the install must be removable
    for name in dirs + files:
      os.chmod(os.path.join(root, name), 0o755 if name in dirs else 0o644)
  os.chmod(tmp, 0o755)
  shutil.rmtree(DEST, ignore_errors=True)
  os.rename(tmp, DEST)
  return True


if __name__ == "__main__":
  ok = build(sys.argv[1] if len(sys.argv) > 1 else None)
  print("reference installed in" if ok else "no reference source readable; nothing installed in", DEST)
