"""Biosample groups: epilogos on column subsets of one matrix.

A group file (`--groups`) has one group per line, `name<TAB>columns`: columns is a comma-separated list of 1-based
biosample numbers and inclusive ranges a-b (biosample 1 is the first label field of a row).  Blank lines and lines
starting with # are ignored.  A group's columns are taken in ascending matrix order, whatever order they are listed in
(what `cut -f` produces), and groups may overlap.

Every stage of the CLI is a function of a shard's per-bin counts or of its label matrix, so a group run needs neither a
matrix directory per group nor a parse per group: the file is parsed and uploaded once (session.Shard), the counts of all
groups come from one epi_group_counts pass over the device matrix, and a group's label matrix (S3, the permutation-replay
null) is gathered from the device matrix.  GroupView presents one group, or one pair of groups for a comparison, with the
interface of session.Shard that the stage drivers use.
"""
import re
from pathlib import Path

import numpy as np

MAX_GROUPS = 64
_NAME = re.compile(r"[A-Za-z0-9._-]+\Z")
_TOKEN = re.compile(r"([0-9]+)(?:-([0-9]+))?\Z")


class GroupFileError(ValueError):
    """A group file that cannot be used; the message is the CLI's `ERROR:` line."""


class GroupSet:
    """The groups of one run, in file order: names and 0-based ascending column arrays."""

    def __init__(self, names, columns):
        self.names = list(names)
        self.columns = [np.asarray(c, dtype=np.int64) for c in columns]
        self.index = {n: i for i, n in enumerate(self.names)}
        self.key = tuple((n, tuple(int(v) for v in c)) for n, c in zip(self.names, self.columns))

    def __len__(self):
        return len(self.names)

    def check_width(self, cols, file):
        """Every column of every group must exist in an input file of `cols` biosamples."""
        for name, c in zip(self.names, self.columns):
            if len(c) and c[-1] >= cols:
                raise ValueError("group '{}' uses biosample {}, but {} has {} biosamples".format(name, int(c[-1]) + 1,
                                                                                            file, cols))

    def select(self, a, b=None):
        """One group (single mode) or the comparison a vs b (paired mode)."""
        return Selection(self, a, b)

    def select_multi(self, names):
        """The multi-group comparison of the named (disjoint) groups (paired mode, --multigroup)."""
        return Selection(self, names[0], multi=tuple(names))


class Selection:
    """One group, a comparison a vs b, or a multi-group comparison of the groups `multi` (its first group is `a`)."""

    def __init__(self, groupset, a, b=None, multi=None):
        self.groupset, self.a, self.b, self.multi = groupset, a, b, multi

    @property
    def paired(self):
        """Whether the selection compares groups: the stage drivers then take the file as their second file too."""
        return self.b is not None or self.multi is not None


def parseGroups(path):
    """The GroupSet of a group file; raises GroupFileError with the message of the first problem."""
    path = Path(path)
    try:
        text = path.read_text()
    except OSError as exc:
        raise GroupFileError("ERROR: [--groups] cannot read {}: {}".format(path, exc.strerror or exc))
    names, columns = [], []
    for n, raw in enumerate(text.splitlines(), start=1):
        line = raw.rstrip("\r")
        if not line.strip() or line.lstrip().startswith("#"):
            continue
        fields = line.split("\t")
        if len(fields) != 2:
            raise GroupFileError("ERROR: [--groups] line {}: expected 'name<TAB>columns', got {!r}".format(n, line))
        name, spec = fields[0].strip(), fields[1].strip()
        if not _NAME.match(name):
            raise GroupFileError("ERROR: [--groups] line {}: group name {!r} must match [A-Za-z0-9._-]+".format(n, name))
        if name in names:
            raise GroupFileError("ERROR: [--groups] line {}: group name '{}' is used twice".format(n, name))
        cols = []
        for tok in (t.strip() for t in spec.split(",")):
            if tok == "":
                continue
            m = _TOKEN.match(tok)
            if not m or int(m.group(1)) < 1 or (m.group(2) is not None and int(m.group(2)) < int(m.group(1))):
                raise GroupFileError("ERROR: [--groups] line {}: {!r} is not a biosample number (from 1) or a range a-b "
                                     "with a <= b".format(n, tok))
            lo = int(m.group(1))
            hi = int(m.group(2)) if m.group(2) is not None else lo
            cols.extend(range(lo, hi + 1))
        if not cols:
            raise GroupFileError("ERROR: [--groups] line {}: group '{}' has no columns".format(n, name))
        ordered = np.sort(np.asarray(cols, dtype=np.int64))
        dup = ordered[1:][ordered[1:] == ordered[:-1]]
        if len(dup):
            raise GroupFileError("ERROR: [--groups] line {}: group '{}' lists biosample {} more than once".format(
                n, name, int(dup[0])))
        if len(names) == MAX_GROUPS:
            raise GroupFileError("ERROR: [--groups] more than {} groups in {}".format(MAX_GROUPS, path))
        names.append(name)
        columns.append(ordered - 1)
    if not names:
        raise GroupFileError("ERROR: [--groups] no group in {}".format(path))
    return GroupSet(names, columns)


def parseMultigroups(specs, groupset):
    """`--multigroup A,B,C` values -> [(A, B, C)]; raises GroupFileError with the first problem, checked in this order
    over all values: an unknown name, a name listed twice, fewer than 2 names, two groups sharing a biosample."""
    lists = [[n.strip() for n in spec.split(",") if n.strip()] for spec in specs]
    for names in lists:
        for n in names:
            if n not in groupset.index:
                raise GroupFileError("ERROR: [--multigroup] group '{}' is not defined in the group file".format(n))
    for spec, names in zip(specs, lists):
        dup = [n for i, n in enumerate(names) if n in names[:i]]
        if dup:
            raise GroupFileError("ERROR: [--multigroup] {!r} lists group '{}' twice".format(spec, dup[0]))
    for spec, names in zip(specs, lists):
        if len(names) < 2:
            raise GroupFileError("ERROR: [--multigroup] {!r} names fewer than 2 groups".format(spec))
    for names in lists:
        for i, a in enumerate(names):
            for b in names[i + 1:]:
                shared = np.intersect1d(groupset.columns[groupset.index[a]], groupset.columns[groupset.index[b]])
                if len(shared):
                    raise GroupFileError("ERROR: [--multigroup] groups '{}' and '{}' share biosample {}".format(
                        a, b, int(shared[0]) + 1))
    return [tuple(names) for names in lists]


def parseComparisons(specs, groupset):
    """`--compare A:B` values -> [(A, B)]; raises GroupFileError."""
    out = []
    for spec in specs:
        parts = spec.split(":")
        if len(parts) != 2 or not parts[0] or not parts[1]:
            raise GroupFileError("ERROR: [--compare] {!r} is not of the form A:B".format(spec))
        a, b = parts
        for g in (a, b):
            if g not in groupset.index:
                raise GroupFileError("ERROR: [--compare] group '{}' is not defined in the group file".format(g))
        if a == b:
            raise GroupFileError("ERROR: [--compare] {!r} compares a group with itself".format(spec))
        out.append((a, b))
    return out


class GroupColumns:
    """The label matrix of one group of a shard, shaped like the matrix a reader would give for that group's column-subset
    file.  A compute backend takes it to the device with device_matrix() (a gather from the shard's device matrix);
    np.asarray gives the host matrix."""

    def __init__(self, shard, columns):
        self._shard, self._columns = shard, columns
        self.shape = (shard.states_a.shape[0], len(columns))

    def device_matrix(self):
        return group_matrix(self._shard, self._columns)

    def head(self, n):
        """The first n rows, on the host."""
        return self._shard.states_a[:n][:, self._columns]

    def __array__(self, dtype=None, copy=None):
        m = self._shard.states_a[:, self._columns]
        return m if dtype is None else m.astype(dtype)


def group_matrix(shard, columns):
    """The columns of a shard's matrix, gathered from its device copy (the file is not parsed or uploaded again)."""
    return shard.backend.gather_columns(shard.states_device(), shard.states_a.shape[1], columns)


def group_counts(shard, groupset):
    """Counts of every group of the set over the shard's rows, indexed by group: one epi_group_counts pass per shard,
    kept with the shard's own counts."""
    key = ("groups", groupset.key)
    if key not in shard._counts:
        groupset.check_width(shard.states_a.shape[1], shard.file)
        shard._counts[key] = shard.backend.group_counts(shard.states_device(), shard.states_a.shape[1], shard.num_states,
                                                        groupset.columns)
    return shard._counts[key]


class GroupView:
    """One group (or the pair of a comparison) of a session.Shard, with the Shard interface of the stage drivers."""

    def __init__(self, shard, selection):
        self._shard, self.selection = shard, selection
        gs = selection.groupset
        gs.check_width(shard.states_a.shape[1], shard.file)
        if selection.multi is not None:
            self._idx = [gs.index[n] for n in selection.multi]
            self.sizes = [len(gs.columns[i]) for i in self._idx]
            self.states_a = GroupColumns(shard, np.sort(np.concatenate([gs.columns[i] for i in self._idx])))
            self.states_b = None
            self._all = self._dev = None
            return
        self._ia = gs.index[selection.a]
        self._ib = gs.index[selection.b] if selection.paired else None
        self.states_a = GroupColumns(shard, gs.columns[self._ia])
        self.states_b = GroupColumns(shard, gs.columns[self._ib]) if selection.paired else None
        self._all = None
        self._dev = None

    def __getattr__(self, name):          # rows, locations, reader: those of the shard
        return getattr(self._shard, name)

    @property
    def paired(self):
        return self.selection.paired

    @property
    def width(self):
        if self.selection.multi is not None:
            return self.states_a.shape[1]
        return self.states_a.shape[1] + (self.states_b.shape[1] if self.paired else 0)

    def group_blocks(self):
        """Counts of the groups of a multi-group comparison, int16 [G, rows, K], in the order they were named."""
        import torch
        cnt = group_counts(self._shard, self.selection.groupset)
        return torch.stack([cnt[i] for i in self._idx])

    def counts(self, which="all"):
        cnt = group_counts(self._shard, self.selection.groupset)
        if self.selection.multi is not None:          # "all": the union of the groups, the background's counts
            if self._all is None:
                self._all = self._shard.backend.add_counts(cnt[self._idx[0]], cnt[self._idx[1]])
                for i in self._idx[2:]:
                    self._all = self._shard.backend.add_counts(self._all, cnt[i])
            return self._all
        if which == "b":
            return cnt[self._ib]
        if which == "a" or not self.paired:
            return cnt[self._ia]
        if self._all is None:
            self._all = self._shard.backend.add_counts(cnt[self._ia], cnt[self._ib])
        return self._all

    def grouped(self):
        """The columns of a multi-group comparison group after group, in the order the groups were named: the matrix
        whose consecutive column slices of `sizes` are the groups (the region null's identity split)."""
        gs = self.selection.groupset
        return GroupColumns(self._shard, np.concatenate([gs.columns[i] for i in self._idx]))

    def combined(self):
        if self.selection.multi is not None:
            return self.states_a
        gs = self.selection.groupset
        cols = gs.columns[self._ia] if not self.paired else np.concatenate((gs.columns[self._ia], gs.columns[self._ib]))
        return GroupColumns(self._shard, cols)

    def states_device(self):
        if self._dev is None:
            self._dev = self.combined().device_matrix()
        return self._dev


def view(shard, selection):
    """The GroupView of a selection of a shard, kept with the shard (its gathered matrix is reused by later stages)."""
    key = (selection.groupset.key, selection.a, selection.b, selection.multi)
    if key not in shard._views:
        shard._views[key] = GroupView(shard, selection)
    return shard._views[key]
