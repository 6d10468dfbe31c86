"""Per-process residency of parsed inputs and per-bin counts.

The reference re-parses every input file in every stage and in every worker (helpers.py:152-155).  Here the
rank's row range of a file is parsed once, packed to int8, counted once on the GPU, and the device-resident
counts (2K bytes per bin) are reused by the score stage of the same process.
"""
import os
import zlib
from pathlib import Path

import numpy as np

from . import dist, helpers

_backend = None
_cache = {}

# In-process hand-over of the score stage to the region-of-interest stage.  The reference passes the scores of every file
# through temp_scores_<tag>_<file>.npz (scores.py:166-169), which the ROI stage reads and deletes (roiSingle.py:43-76).  When
# both stages run in THIS process (the CLI, run.run_stages) the arrays are handed over in memory instead: the file would
# be written, read back and removed within seconds (0.3-0.6 s of a 2 s run at 400 k bins x 833).  Stand-alone calls of
# scores.main still write the file, and EPILOGOS_B200_KEEP_TEMP=1 forces it everywhere.
handover = {}              # str(path of the temp_scores npz that was not written) -> dict(chrName, scoreArr, chrom, start, end)
handover_enabled = False


def get_backend(backend=None):
    global _backend
    if backend is not None:
        return backend
    if _backend is None:
        from .backend import CudaBackend
        _backend = CudaBackend()
    return _backend


def one_reader():
    """With the rows of a file sharded over several ranks, ONE rank reads the file and deals the row ranges to the others
    (EPILOGOS_B200_READ=deal), instead of every rank inflating and parsing the whole file to keep its 1/N of the rows
    (EPILOGOS_B200_READ=redundant: the behaviour up to round 2, no exchange of rows).  Unset: deal over gloo, where the
    exchange is covered by the CPU suite; over NCCL the exchange (device tensors, point-to-point) was written without a GPU
    at hand, so it stays opt-in until tools/mgpu_check.py has passed with it on a multi-GPU box."""
    mode = os.environ.get("EPILOGOS_B200_READ", "")
    if mode in ("deal", "redundant"):
        return mode == "deal"
    try:
        import torch.distributed as td
        return td.is_available() and td.is_initialized() and td.get_backend() == "gloo"
    except Exception:
        return False


def reader_of(file1, world):
    """The rank that reads a file when nobody assigned one: spread by file name, the same on every rank."""
    return zlib.crc32(Path(file1).name.encode()) % world


def _pack_locations(loc):
    """Locations in a form that pickles in no time: coordinates as they are, chromosome names run-length encoded."""
    chrom = np.asarray(loc["chrom"], dtype=object)
    n = len(chrom)
    if n == 0:
        return dict(start=loc["start"], end=loc["end"], names=[], runs=[])
    change = np.flatnonzero(chrom[1:] != chrom[:-1]) + 1
    first = np.concatenate(([0], change))
    length = np.diff(np.concatenate((first, [n])))
    return dict(start=np.asarray(loc["start"]), end=np.asarray(loc["end"]), names=[str(chrom[i]) for i in first],
                runs=[int(v) for v in length])


def _unpack_locations(packed):
    n = sum(packed["runs"])
    chrom = np.empty(n, dtype=object)
    table = []                                     # distinct names in order of first appearance, as the native parser lists them
    cid = np.empty(n, dtype=np.int32)
    at = 0
    for name, run in zip(packed["names"], packed["runs"]):
        if name not in table:
            table.append(name)
        chrom[at:at + run] = name
        cid[at:at + run] = table.index(name)
        at += run
    return dict(chrom=chrom, start=packed["start"], end=packed["end"], chrom_id=cid,
                chrom_names=b"".join(t.encode() + b"\0" for t in table) or b"\0")


class Shard:
    """The rows [lo, hi) of one input file (or file pair) owned by this rank."""

    def __init__(self, file1, file2, num_states, backend, rank=0, world=0, reader=None, exchange=True):
        self.backend = get_backend(backend)
        self.num_states = num_states
        if not Path(file1).is_file():
            raise FileNotFoundError(str(file1))
        pinned = getattr(self.backend, "name", "") == "cuda"
        split = (rank, world) if world else (dist.rank(), dist.world_size())
        self.file = Path(file1)
        self._counts = {}
        self._states_dev = None
        self._views = {}              # groups.GroupView of this shard, by selection
        self.reader = None            # the rank that read the file when the rows were dealt (one_reader); else None
        self.loc_full = None          # locations of ALL rows, on rank 0, when the rows were dealt
        if split[1] > 1 and one_reader():
            # ---- one reader per file: no file is inflated or parsed more than once, whatever the number of ranks
            self.reader = reader_of(file1, split[1]) if reader is None else int(reader)
            self._split, self._pinned, self._paired = split, pinned, str(file2) != "null"
            self._full = None
            if split[0] == self.reader:
                try:
                    loc, a, total = helpers.read_matrix(file1, None, want_locations=True, num_states=num_states,
                                                        pinned=pinned, return_total=True)
                    b = None
                    if self._paired:
                        _, b = helpers.read_matrix(file2, None, want_locations=False, num_states=num_states, pinned=pinned)
                        if b.shape[0] != a.shape[0]:
                            raise ValueError("paired input files must have the same number of rows")
                    self._full = (loc, a, b, total)
                except Exception as exc:           # the other ranks wait in exchange(): tell them instead of leaving
                    self._full = exc
            if exchange:
                self.exchange()
            return
        # ---- every rank reads the file itself.  One pass: the row count comes out of the parse, this rank's range is cut
        # from the parsed rows
        self.loc, self.states_a, self.total_rows = helpers.read_matrix(file1, None, want_locations=True,
                                                                       num_states=num_states, pinned=pinned,
                                                                       split=split, return_total=True)
        self.lo, self.hi = helpers.splitRows(self.total_rows, split[1])[split[0]]
        rows = (self.lo, self.hi)
        self.states_b = None
        if str(file2) != "null":
            _, self.states_b = helpers.read_matrix(file2, rows, want_locations=False, num_states=num_states)
            if self.states_b.shape[0] != self.states_a.shape[0]:
                raise ValueError("paired input files must have the same number of rows")

    def exchange(self):
        """Collective (every rank, same order of files): the reader announces the shape, deals the row ranges of
        helpers.splitRows to the ranks and hands the locations to rank 0, which writes the outputs."""
        import torch.distributed as td
        rank, world = self._split
        meta = [None]
        if rank == self.reader:
            if isinstance(self._full, Exception):
                meta = [("error", type(self._full).__name__, str(self._full))]
            else:
                loc, a, b, total = self._full
                meta = [(int(total), int(a.shape[1]), int(b.shape[1]) if b is not None else -1)]
        td.broadcast_object_list(meta, src=self.reader)
        if meta[0][0] == "error":                  # every rank fails the same way, as when each read the file itself
            if rank == self.reader:
                raise self._full
            kinds = {"ValueError": ValueError, "FileNotFoundError": FileNotFoundError}
            raise kinds.get(meta[0][1], RuntimeError)("rank %d could not read the input: %s" % (self.reader, meta[0][2]))
        total, cols_a, cols_b = meta[0]
        ranges = helpers.splitRows(total, world)
        self.total_rows = total
        self.lo, self.hi = ranges[rank]
        def pitched(m, pitch):
            """The [rows, pitch] buffer behind a matrix of read_matrix (it is a view of one), else a pitched copy."""
            base = m.base
            if (isinstance(base, np.ndarray) and base.dtype == np.int8 and base.ndim == 2 and base.flags.c_contiguous
                    and base.shape == (m.shape[0], pitch) and (m.size == 0 or m.ctypes.data == base.ctypes.data)):
                return base
            out = np.zeros((m.shape[0], pitch), dtype=np.int8)
            out[:, :m.shape[1]] = m
            return out
        pitch_a, pitch_b = helpers.pitch_for(max(cols_a, 1)), helpers.pitch_for(max(cols_b, 1))
        full_a = pitched(a, pitch_a) if rank == self.reader else None
        full_b = pitched(b, pitch_b) if rank == self.reader and b is not None else None
        self.states_a = dist.deal_rows(full_a, ranges, self.reader, pitch_a, self._pinned)[:, :cols_a]
        self.states_b = None
        if cols_b >= 0:
            self.states_b = dist.deal_rows(full_b, ranges, self.reader, pitch_b, self._pinned)[:, :cols_b]
        # locations: only the writing rank needs them
        self.loc = None
        if self.reader == 0:
            if rank == 0:
                self.loc_full = loc                # with the parser's chromosome ids: the writer needs no np.unique
        else:
            box = [_pack_locations(loc)] if rank == self.reader else [None]
            if rank == self.reader:
                td.send_object_list(box, dst=0)
            elif rank == 0:
                td.recv_object_list(box, src=self.reader)
                self.loc_full = _unpack_locations(box[0])
        self._full = None

    @property
    def paired(self):
        return self.states_b is not None

    @property
    def width(self):
        """Biosamples of the matrix the expected table is computed over: the union of both groups in paired
        mode (helpers.py:173-179)."""
        return self.states_a.shape[1] + (self.states_b.shape[1] if self.paired else 0)

    def combined(self):
        return self.states_a if not self.paired else np.concatenate((self.states_a, self.states_b), axis=1)

    def counts(self, which="all"):
        """Per-bin counts of the whole matrix ("all": the union [A | B] in paired mode) or of one group."""
        if which not in self._counts:
            if which == "all" and self.paired:
                self._counts[which] = self.backend.add_counts(self.counts("a"), self.counts("b"))
            else:
                m = self.states_b if which == "b" else self.states_a
                self._counts[which] = self.backend.counts(m, self.num_states)
        return self._counts[which]

    def states_device(self):
        if self._states_dev is None:
            self._states_dev = self.backend.states_to_device(self.combined())
        return self._states_dev


def _key(file1, file2):
    p1 = Path(file1).resolve()
    st = p1.stat()
    return (str(p1), st.st_mtime_ns, st.st_size, str(file2), dist.rank(), dist.world_size())


_keep = 4


def load_shard(file1, file2, num_states, backend=None, keep=None, group=None):
    """The cached Shard of a file (pair).  With `group` (a groups.Selection) the shard of file1 alone is loaded and the
    view of that group, or of that comparison of two groups, is returned; file2 is then not read."""
    if group is not None:
        from . import groups
        return groups.view(load_shard(file1, "null", num_states, backend, keep), group)
    key = _key(file1, file2)
    if key not in _cache:
        while len(_cache) >= (keep or _keep):
            _cache.pop(next(iter(_cache)))
        if dist.world_size() > 1 and one_reader():
            from . import _lib
            _lib.call("epi_reader_concurrency", 1, 1)      # one rank reads this file: it may use the whole host
            try:
                _cache[key] = Shard(file1, file2, num_states, backend)
            finally:
                _lib.call("epi_reader_concurrency", 0, 0)
        else:
            _cache[key] = Shard(file1, file2, num_states, backend)
    return _cache[key]


def prefetch(pairs, num_states, backend=None, workers=None):
    """Parse the input files concurrently and once, before the stages run.  The reference parses every file again in every
    stage and worker; the native packer (csrc/hostio.cu) releases the GIL and gives every file its share of the cores
    (inflate | parse threads), so a whole-genome directory of per-chromosome files is read in the time of its largest
    files instead of their sum.  With the rows sharded over several ranks the files are dealt to the ranks as READERS by
    size (largest first, round robin); every reader then deals the row ranges of its files to all ranks, so no file is
    read twice and every rank still holds 1/N of every file.  The cache is sized to hold every file, so the score stage
    re-uses the parsed matrices and the device-resident counts of the expected stage."""
    from concurrent.futures import ThreadPoolExecutor
    from . import _lib
    global _keep
    pairs = list(pairs)
    _keep = max(_keep, len(pairs) + 1)
    todo = [(f, f2) for f, f2 in pairs if _key(f, f2) not in _cache]
    if not todo:
        return
    be = get_backend(backend)
    rank, world = dist.rank(), dist.world_size()          # resolved on the calling thread
    dealt = world > 1 and one_reader()
    readers = [None] * len(todo)
    mine = len(todo)
    if dealt:
        order = sorted(range(len(todo)), key=lambda i: (-Path(todo[i][0]).stat().st_size, str(todo[i][0])))
        for j, i in enumerate(order):
            readers[i] = j % world
        mine = sum(1 for r in readers if r == rank)
    workers = workers or max(1, min(max(mine, 1), (os.cpu_count() or 2) // 2))
    # every reader takes its share of the cores from the start; with dealt files only min(world, files) ranks read at all
    _lib.call("epi_reader_concurrency", int(min(workers, max(mine, 1))), int(min(world, len(todo))) if dealt else 0)
    try:
        with ThreadPoolExecutor(max_workers=workers) as pool:
            shards = list(pool.map(lambda a: Shard(a[0][0], a[0][1], num_states, be, rank=rank, world=world, reader=a[1],
                                                   exchange=False), zip(todo, readers)))
    finally:
        _lib.call("epi_reader_concurrency", 0, 0)
    for (f, f2), sh in zip(todo, shards):
        if sh.reader is not None:
            sh.exchange()                                  # collectives: calling thread, same file order on every rank
        _cache[_key(f, f2)] = sh


def clear():
    _cache.clear()
