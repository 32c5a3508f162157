#!/usr/bin/env python3
"""Stage the UNMODIFIED reference into ``oracle/_ref/`` (git-ignored; it travels with the tree).

The reference (lvclark/tagdigger) is pure, stdlib-only Python: there is nothing to compile.  The
repository does not ship it; given a checkout of it in the environment variable
``TAGDIGGER_REFERENCE``, the files that make up the reference's counting path are copied -- byte
for byte, by this recipe only -- into ``oracle/_ref/``, so that the tree carries them to where it
runs like its own built ``.so`` files.  Nothing here is product source: ``oracle/_ref/`` is listed
in ``.gitignore`` and is imported only by ``bench.py --impl reference`` / the ``cpu_baseline`` leg
and by ``tests/`` (the live comparisons with the reference, skipped where nothing is staged).

    TAGDIGGER_REFERENCE=<checkout> python oracle/stage_ref.py            # copy + write MANIFEST.json
    TAGDIGGER_REFERENCE=<checkout> python oracle/stage_ref.py --check    # verify an existing stage

TEST / BENCH INFRASTRUCTURE ONLY.
"""

import hashlib
import json
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.environ.get("TAGDIGGER_REFERENCE", "")
DST = os.path.join(HERE, "_ref")
# the library, the two scripts that drive the counting path (tagdigger_script.py:123-133) and
# the splitter script of the two-stage flow (barcode_splitter_script.py:8-36)
FILES = ["tagdigger_fun.py", "tagdigger_script.py", "barcode_splitter_script.py"]


def sha256(path):
    h = hashlib.sha256()
    with open(path, "rb") as fh:
        for block in iter(lambda: fh.read(1 << 20), b""):
            h.update(block)
    return h.hexdigest()


def staged():
    """True when oracle/_ref holds every file its manifest lists, unchanged."""
    try:
        with open(os.path.join(DST, "MANIFEST.json")) as fh:
            man = json.load(fh)
        return all(sha256(os.path.join(DST, f)) == d for f, d in man["sha256"].items()) and \
            set(man["sha256"]) == set(FILES)
    except (OSError, ValueError, KeyError):
        return False


def stage():
    if not SRC or not os.path.isdir(SRC):
        return staged()
    os.makedirs(DST, exist_ok=True)
    digests = {}
    for f in FILES:
        shutil.copyfile(os.path.join(SRC, f), os.path.join(DST, f))
        os.chmod(os.path.join(DST, f), 0o644)
        digests[f] = sha256(os.path.join(DST, f))
        assert digests[f] == sha256(os.path.join(SRC, f))
    with open(os.path.join(DST, "MANIFEST.json"), "w") as fh:
        json.dump({"source": SRC, "note": "unmodified copies of lvclark/tagdigger (GPL-3); bench/test use only",
                   "sha256": digests}, fh, indent=1, sort_keys=True)
    return True


def check():
    if not staged():
        return False
    if SRC and os.path.isdir(SRC):
        with open(os.path.join(DST, "MANIFEST.json")) as fh:
            man = json.load(fh)
        return all(sha256(os.path.join(SRC, f)) == d for f, d in man["sha256"].items())
    return True


def import_ref():
    """The staged reference's ``tagdigger_fun`` module (None when nothing is staged)."""
    if not staged():
        return None
    import importlib.util
    import warnings
    spec = importlib.util.spec_from_file_location("tagdigger_ref_fun", os.path.join(DST, "tagdigger_fun.py"))
    mod = importlib.util.module_from_spec(spec)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")          # SyntaxWarning for '\d' at tagdigger_fun.py:772-773
        spec.loader.exec_module(mod)
    return mod


if __name__ == "__main__":
    if "--check" in sys.argv:
        ok = check()
        print("oracle/_ref:", "ok" if ok else "missing or modified")
        sys.exit(0 if ok else 1)
    print("oracle/_ref staged" if stage() else "nothing staged: TAGDIGGER_REFERENCE names no directory")
