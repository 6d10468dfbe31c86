"""Build the UNMODIFIED reference into a form that can travel with the source tree.

TEST / BENCHMARK INFRASTRUCTURE ONLY.  The reference (meuleman/epilogos) is pure Python, so "building" it means compiling:
the modules the scoring path imports are byte-compiled with py_compile straight from a checkout of the reference named by
the environment variable EPILOGOS_REFERENCE into oracle/_ref/epilogos/*.pyc (sourceless layout, importable as the package
`epilogos`).  No reference SOURCE is copied anywhere; oracle/_ref/ holds build outputs only and is git-ignored, so it can
be shipped with a built tree like the .so and `bench.py --impl reference` / `cpu_baseline` can time the reference's real
`expected.main -> expectedCombination.main -> scores.main` path (TSV.gz parse and gz write included, run.py:191-303) on a
host with the same CPython.  Without EPILOGOS_REFERENCE nothing is staged, and whatever needs the reference skips or falls
back to the oracle's port.

    EPILOGOS_REFERENCE=/path/to/epilogos python -m oracle.stage_reference     # also run by __graft_entry__.build()

A MANIFEST with the sha256 of every SOURCE file that was compiled is written so that a run can state exactly what it timed.
"""
import hashlib
import json
import os
import py_compile
import shutil
import sys
from pathlib import Path

SOURCE = Path(os.environ["EPILOGOS_REFERENCE"]) if os.environ.get("EPILOGOS_REFERENCE") else None
DEST = Path(__file__).resolve().parent / "_ref"

# the modules the scoring path imports (expected / expectedCombination / scores -> helpers -> filter_regions)
FILES = ["epilogos/__init__.py", "epilogos/expected.py", "epilogos/expectedCombination.py", "epilogos/scores.py",
         "epilogos/helpers.py", "epilogos/filter_regions.py"]


def source_available():
    """True when EPILOGOS_REFERENCE names a readable checkout of the reference."""
    try:
        return SOURCE is not None and (SOURCE / "epilogos" / "scores.py").is_file()
    except OSError:                                   # e.g. a directory this user may not enter
        return False


def staged_root():
    """Directory to put on sys.path to import the reference: the EPILOGOS_REFERENCE checkout when there is one, else the
    byte-compiled build under oracle/_ref, else None.  EPI_REF_FORCE_STAGED=1 prefers the build (tests)."""
    built = (DEST / "epilogos" / "scores.pyc").is_file()
    if built and os.environ.get("EPI_REF_FORCE_STAGED"):
        return DEST
    if source_available():
        return SOURCE
    return DEST if built else None


def stage(verbose=True):
    if not source_available():
        if verbose:
            print("stage_reference: EPILOGOS_REFERENCE does not name a checkout of the reference, nothing built")
        return None
    if (DEST / "epilogos").exists():
        shutil.rmtree(DEST / "epilogos")
    (DEST / "epilogos").mkdir(parents=True)
    manifest = {}
    for rel in FILES:
        src = SOURCE / rel
        dst = DEST / (rel + "c")                      # epilogos/scores.pyc: sourceless import layout
        if not src.is_file():
            raise FileNotFoundError(src)
        import warnings
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")           # SyntaxWarnings of the reference's own regex literals
            py_compile.compile(str(src), cfile=str(dst), dfile="<reference>/" + rel, doraise=True, optimize=0, quiet=1)
        manifest[rel] = hashlib.sha256(src.read_bytes()).hexdigest()
    (DEST / "MANIFEST.json").write_text(json.dumps({"source": str(SOURCE), "python": sys.version.split()[0],
                                                   "what": "py_compile of the listed reference sources (sha256 of each source)",
                                                   "sha256": manifest}, indent=1))
    if verbose:
        print("stage_reference: %d modules byte-compiled -> %s" % (len(manifest), DEST))
    return DEST


if __name__ == "__main__":
    stage()
