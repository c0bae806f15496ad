#!/usr/bin/env python
"""Copies the three files of the UNMODIFIED reference that the hot path needs into the git-ignored baseline/_ref/
(BASELINE.md section 4.1), so that the reference itself can be timed -- and used as a second checker -- by
bench.py's CPU arm.  Nothing under baseline/_ref/ is tracked or imported by the product; only bench.py's CPU arm
uses it, through ``import_reference()`` below, and reports it unavailable when nothing was vendored.

    python baseline/vendor_ref.py <checkout of AnnaLew/pangenomix>/pangenomix
"""
import os
import shutil
import sys
import types

HERE = os.path.dirname(os.path.abspath(__file__))
REF_DST = os.path.join(HERE, "_ref", "pangenomix")
FILES = ["__init__.py", "pangenome_analysis.py", "sparse_utils.py"]


def vendor(src):
    """Copies FILES from ``src``, the reference's package directory."""
    os.makedirs(REF_DST, exist_ok=True)
    for name in FILES:
        shutil.copyfile(os.path.join(src, name), os.path.join(REF_DST, name))


def available():
    return all(os.path.exists(os.path.join(REF_DST, name)) for name in FILES)


def import_reference():
    """(pangenome_analysis, sparse_utils) of the vendored reference.  statsmodels (imported at
    pangenome_analysis.py:18, used only at :380, off the hot path) is absent from the image and stubbed."""
    if not available():
        raise ImportError("baseline/_ref is empty: run baseline/vendor_ref.py <reference package directory>")
    import importlib.util
    for name in ("statsmodels", "statsmodels.stats"):
        sys.modules.setdefault(name, types.ModuleType(name))
    mods = {}
    # loaded under a private package name so that it cannot shadow the drop-in ``pangenomix`` shim of this repo
    pkg = types.ModuleType("pgx_reference")
    pkg.__path__ = [REF_DST]
    sys.modules["pgx_reference"] = pkg
    saved = sys.modules.get("pangenomix"), sys.modules.get("pangenomix.sparse_utils")
    for name in ("sparse_utils", "pangenome_analysis"):
        spec = importlib.util.spec_from_file_location("pgx_reference." + name, os.path.join(REF_DST, name + ".py"))
        mod = importlib.util.module_from_spec(spec)
        sys.modules["pgx_reference." + name] = mod
        if name == "sparse_utils":
            # the reference's pangenome_analysis does ``import pangenomix.sparse_utils`` (:22): give it its own
            fake = types.ModuleType("pangenomix")
            fake.sparse_utils = mod
            sys.modules["pangenomix"] = fake
            sys.modules["pangenomix.sparse_utils"] = mod
        spec.loader.exec_module(mod)
        mods[name] = mod
    for key, old in zip(("pangenomix", "pangenomix.sparse_utils"), saved):
        if old is None:
            sys.modules.pop(key, None)
        else:
            sys.modules[key] = old
    return mods["pangenome_analysis"], mods["sparse_utils"]


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit("usage: python baseline/vendor_ref.py <reference package directory>")
    vendor(sys.argv[1])
    print("vendored into %s" % REF_DST)
