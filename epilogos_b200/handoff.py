"""The trip of each input file's score-stage result (step 3) to the regions-of-interest stage (step 4).

A record is a dict: chrName, chrom, start, end and the kind's keys (FILES; paired mode adds distance and max_diff in
memory only, from files step 4 reduces the delta text).  When step 4 runs next in this process (session.handover_enabled)
the record stays in memory, device tensors included; otherwise, and always with EPILOGOS_B200_KEEP_TEMP set, it goes
through temp_<prefix>_<tag>_<file>.npz files.  temp_scores, temp_nullDistances and temp_quiescence are the reference's
own format (scores.py:166-169, 234-247); the others are read by the python -m epilogos_b200.roi_* entry points.
"""
import glob
import os
from pathlib import Path

import numpy as np

from . import dist, helpers, region_null, session, writer

LOCATION = ("chrom", "start", "end")           # one object array [rows, 3], as writer.location_array builds it
_PERMUTATIONS = (("exceedances", "exceedances", np.uint32), ("permutations", "permutations", np.int64))
_REGION = ("regionNull", (("maxima", "region_maxima", np.int64), ("window", "region_window", np.int64),
                          ("permutations", "region_permutations", np.int64)))

# kind -> its files: (prefix, ((npz key, record key, dtype), ...)).  Every file also holds chrName as a 1-element string
# array.  A key is written when the record has it, a file when it has any such key; step 4 finds a file's results by the
# first file of its kind.
FILES = {
    "scores": (("scores", (("scoreArr", "scoreArr", np.float32), ("locationArr", LOCATION, object))),),
    "paired": (("nullDistances", (("nullDistances", "null", np.float32),)),
               ("quiescence", (("quiescenceArr", "quiescence", np.bool_),)),
               ("permutations", _PERMUTATIONS),
               _REGION),
    "multigroup": (("multigroup", (("groups", "groups", str), ("t", "t", np.float64), ("group", "group", np.uint8),
                                   ("state", "state", np.uint8), ("sign", "sign", np.int8), ("chrom", "chrom", str),
                                   ("start", "start", np.int64), ("end", "end", np.int64)) + _PERMUTATIONS),
                   _REGION),
}


def record(loc, **parts):
    """A record (rank 0): chrName (the chromosome of the file's first row), the locations of its rows and `parts`."""
    chrom = np.asarray(loc["chrom"], dtype=object)
    return dict(chrName=str(chrom[0]) if len(chrom) else "", chrom=chrom, start=np.asarray(loc["start"], dtype=np.int64),
                end=np.asarray(loc["end"], dtype=np.int64), **parts)


def optional_parts(path, loc, total, exceed, permutations, region, window, region_permutations):
    """The optional keys of a paired or multi-group record of input file `path`.  Collective: every rank gathers its
    exceedance counts; rank 0 gets the dict, the other ranks None."""
    exceed = None if exceed is None else dist.gather_rows(exceed, total)
    if dist.rank() != 0:
        return None
    out = {}
    if exceed is not None:
        out.update(exceedances=exceed, permutations=int(permutations))
    if region is not None:
        region_null.check_one_chromosome(loc["chrom"], path)
        out.update(region_maxima=np.asarray(region.cpu().numpy(), dtype=np.int64), region_window=int(window),
                   region_permutations=int(region_permutations))
    return out


def _host(x):
    return x.cpu().numpy() if hasattr(x, "cpu") else np.asarray(x)


def _pattern(kind, prefix, tag):
    # single mode takes every temp_scores file of the directory, whatever its tag, as the reference's roiSingle does
    return "temp_{}_{}_*.npz".format(prefix, "*" if kind == "scores" else glob.escape(tag))


def publish(kind, out_dir, tag, filename, rec, in_memory=None):
    """Hand `rec` over to step 4 of this process, or write it to its temp files.  `in_memory()` gives the parts that only
    the hand-over carries (from files, step 4 derives them from other outputs of the stage)."""
    if session.handover_enabled and not os.environ.get("EPILOGOS_B200_KEEP_TEMP"):
        session.handover[(kind, Path(out_dir), tag, filename)] = dict(rec, **(in_memory() if in_memory else {}))
        return
    for prefix, keys in FILES[kind]:
        arrays = {}
        for npz_key, key, dtype in keys:
            if key == LOCATION:
                arrays[npz_key] = writer.location_array(rec)
            elif key in rec:
                arrays[npz_key] = _host(rec[key]).astype(dtype, copy=False)
        if arrays:
            helpers.savez_level(Path(out_dir) / "temp_{}_{}_{}.npz".format(prefix, tag, filename),
                                chrName=np.array([rec["chrName"]]), **arrays)


def _read(kind, path):
    """The record of a file of the kind's first prefix, with the keys of the kind's other files of the same input file."""
    first = FILES[kind][0][0]
    rec = {}
    for prefix, keys in FILES[kind]:
        f = path.with_name(path.name.replace("temp_{}_".format(first), "temp_{}_".format(prefix), 1))
        if not f.exists():
            continue
        z = np.load(f, allow_pickle=kind == "scores")
        rec["chrName"] = str(z["chrName"][0])
        for npz_key, key, dtype in keys:
            if npz_key not in z.files:
                continue
            v = z[npz_key]
            if key == LOCATION:
                rec.update(chrom=v[:, 0], start=v[:, 1].astype(np.int64), end=v[:, 2].astype(np.int64))
            elif dtype is str:
                rec[key] = v.astype(object)
            else:
                rec[key] = int(v) if v.ndim == 0 else v
    return rec


def collect(kind, out_dir, tag, from_files=None):
    """The records of this directory and tag in chromosome order (roi.orderChromosomes): those handed over, then those of
    the files of chromosomes not handed over.  exceedances come as numpy uint32 either way.  `from_files(rec, name)`
    completes a record read from temp_<prefix>_<tag>_<name>.npz."""
    from .roi import orderChromosomes
    out_dir = Path(out_dir)
    chunks = {}
    for key in [k for k in session.handover if k[:2] == (kind, out_dir) and (kind == "scores" or k[2] == tag)]:
        rec = session.handover.pop(key)
        chunks[rec["chrName"]] = rec
    first = FILES[kind][0][0]
    for f in sorted(out_dir.glob(_pattern(kind, first, tag))):
        rec = _read(kind, f)
        if rec["chrName"] not in chunks:
            if from_files is not None:
                from_files(rec, f.name[len("temp_{}_{}_".format(first, tag)):-len(".npz")])
            chunks[rec["chrName"]] = rec
    if not chunks:
        raise FileNotFoundError("no score-stage outputs ({}) in {}".format(_pattern(kind, first, tag), out_dir))
    for rec in chunks.values():
        if "exceedances" in rec:
            rec["exceedances"] = _host(rec["exceedances"]).view(np.uint32)
    return [chunks[c] for c in orderChromosomes(list(chunks))]


def remove_temps(kind, out_dir, tag):
    """Remove the kind's temp files of this directory and tag (single mode: of every tag)."""
    for prefix, _ in FILES[kind]:
        for f in Path(out_dir).glob(_pattern(kind, prefix, tag)):
            f.unlink()
