"""Stages the UNMODIFIED reference (visionml/pytracking, /root/reference) into baseline/_ref/ so that it travels to the GPU box
with the gpurun snapshot (baseline/_ref/ is git-ignored, not gpurun-ignored).

The reference has no setup.py / pyproject.toml (it is used from its source tree, INSTALL.md), so "installing" it is copying the
two importable packages `pytracking/` and `ltr/` byte for byte; nothing is edited.  `baseline/ref_env.py` then puts
baseline/_ref on sys.path and installs the out-of-tree compatibility shims (SURVEY.md 8(c)).

    PYTRACKING_REFERENCE=<pytracking checkout> python baseline/stage_reference.py        # idempotent
"""
import hashlib
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.environ.get("PYTRACKING_REFERENCE", "/root/reference")
DST = os.path.join(HERE, "_ref")
PACKAGES = ("pytracking", "ltr")
KEEP_EXT = (".py", ".c", ".h", ".cu", ".cuh", ".md", ".txt", ".json")


def _tree_digest(root):
    h = hashlib.sha256()
    for pkg in PACKAGES:
        for d, _, files in sorted(os.walk(os.path.join(root, pkg))):
            for f in sorted(files):
                if f.endswith(KEEP_EXT):
                    p = os.path.join(d, f)
                    h.update(os.path.relpath(p, root).encode())
                    h.update(open(p, "rb").read())
    return h.hexdigest()


def stage(force=False):
    if not os.path.isdir(os.path.join(SRC, "pytracking")):
        return None
    want = _tree_digest(SRC)
    stamp = os.path.join(DST, "STAGED_FROM")
    if not force and os.path.exists(stamp) and open(stamp).read().split()[-1] == want:
        return DST
    if os.path.isdir(DST):
        shutil.rmtree(DST)
    os.makedirs(DST)
    for pkg in PACKAGES:
        shutil.copytree(os.path.join(SRC, pkg), os.path.join(DST, pkg),
                        ignore=lambda d, names: [n for n in names if not (os.path.isdir(os.path.join(d, n)) or n.endswith(KEEP_EXT))])
    for f in ("LICENSE",):
        if os.path.exists(os.path.join(SRC, f)):
            shutil.copy(os.path.join(SRC, f), os.path.join(DST, f))
    assert _tree_digest(DST) == want, "staged copy differs from the reference"
    with open(stamp, "w") as fh:
        fh.write("visionml/pytracking staged unmodified from %s sha256(tree) %s\n" % (SRC, want))
    return DST


if __name__ == "__main__":
    d = stage(force="--force" in sys.argv)
    print(d if d else "reference tree not found at %s" % SRC)
