"""Build recipe of ``oracle/_ref``: the unmodified reference (grid2op, pure Python) installed next to the oracle.

``B200Backend`` plugs into grid2op, and most tests step real grid2op environments on it or compare it with grid2op's own
suites and bundled grids.  ``build()`` therefore installs the reference's ``grid2op`` package (sources, bundled ``data``,
``data_test`` fixtures and ``tests`` suites) from a reference checkout into ``oracle/_ref/grid2op``; the package finds it
there (``grid2op_b200/_bootstrap.py``) on machines that have no grid2op installed and no checkout.  ``oracle/_ref`` is a
build product and is not tracked.

The checkout is ``$GRID2OP_B200_REF`` when set, else the directory the project's reference checkout is kept in
(``REFERENCE_CHECKOUT``).  Without a checkout an existing ``oracle/_ref`` is kept as it is."""
import os
import shutil
import stat

HERE = os.path.dirname(os.path.abspath(__file__))
DEST = os.path.join(HERE, "_ref")
REFERENCE_CHECKOUT = "/root/reference"


def checkout():
    """-> the reference checkout to install from, or None"""
    for root in (os.environ.get("GRID2OP_B200_REF", ""), REFERENCE_CHECKOUT):
        if root and os.path.isfile(os.path.join(root, "grid2op", "__init__.py")):
            return root
    return None


def build(force: bool = False):
    """Install the reference's grid2op package into oracle/_ref (once; ``force`` re-installs) -> oracle/_ref or None"""
    if os.path.isfile(os.path.join(DEST, "grid2op", "__init__.py")) and not force:
        return DEST
    src = checkout()
    if src is None:
        return None
    tmp = f"{DEST}.{os.getpid()}.tmp"
    shutil.rmtree(tmp, ignore_errors=True)
    shutil.copytree(os.path.join(src, "grid2op"), os.path.join(tmp, "grid2op"), copy_function=shutil.copyfile,
                    ignore=shutil.ignore_patterns("__pycache__", "*.pyc"))
    for d, _, files in os.walk(tmp):                 # a read-only checkout must not make the install read-only
        for p in [d] + [os.path.join(d, f) for f in files]:
            os.chmod(p, os.stat(p).st_mode | stat.S_IWUSR)
    if os.path.isdir(DEST):
        shutil.rmtree(DEST)
    os.replace(tmp, DEST)
    return DEST


if __name__ == "__main__":
    print(build(force=True))
