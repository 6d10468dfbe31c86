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


def parseGroups(path, flag="--groups"):
    """The GroupSet of a group file; raises GroupFileError with the message of the first problem.  `flag` is the option
    the messages name (the strata file of --strata has the same format)."""
    path = Path(path)
    try:
        text = path.read_text()
    except OSError as exc:
        raise GroupFileError("ERROR: [{}] cannot read {}: {}".format(flag, path, exc.strerror or exc))
    names, columns = [], []
    for n, raw in enumerate(text.splitlines(), start=1):
        line = raw.rstrip("\r")
        if not line.strip() or line.lstrip().startswith("#"):
            continue
        fields = line.split("\t")
        if len(fields) != 2:
            raise GroupFileError("ERROR: [{}] line {}: expected 'name<TAB>columns', got {!r}".format(flag, n, line))
        name, spec = fields[0].strip(), fields[1].strip()
        if not _NAME.match(name):
            raise GroupFileError("ERROR: [{}] line {}: group name {!r} must match [A-Za-z0-9._-]+".format(flag, n, name))
        if name in names:
            raise GroupFileError("ERROR: [{}] line {}: group name '{}' is used twice".format(flag, n, name))
        cols = []
        for tok in (t.strip() for t in spec.split(",")):
            if tok == "":
                continue
            m = _TOKEN.match(tok)
            if not m or int(m.group(1)) < 1 or (m.group(2) is not None and int(m.group(2)) < int(m.group(1))):
                raise GroupFileError("ERROR: [{}] line {}: {!r} is not a biosample number (from 1) or a range a-b "
                                     "with a <= b".format(flag, n, tok))
            lo = int(m.group(1))
            hi = int(m.group(2)) if m.group(2) is not None else lo
            cols.extend(range(lo, hi + 1))
        if not cols:
            raise GroupFileError("ERROR: [{}] line {}: group '{}' has no columns".format(flag, n, name))
        ordered = np.sort(np.asarray(cols, dtype=np.int64))
        dup = ordered[1:][ordered[1:] == ordered[:-1]]
        if len(dup):
            raise GroupFileError("ERROR: [{}] line {}: group '{}' lists biosample {} more than once".format(
                flag, n, name, int(dup[0])))
        if len(names) == MAX_GROUPS:
            raise GroupFileError("ERROR: [{}] more than {} groups in {}".format(flag, MAX_GROUPS, path))
        names.append(name)
        columns.append(ordered - 1)
    if not names:
        raise GroupFileError("ERROR: [{}] no group in {}".format(flag, path))
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


# ---- strata (--strata): null shuffles that move labels only within strata ------------------------------------------------

class Strata:
    """The strata of a run, in file order (a GroupSet of disjoint column sets), and the file they came from."""

    def __init__(self, groupset, path):
        self.groupset, self.path = groupset, str(path)

    def __len__(self):
        return len(self.groupset)

    def summary(self):
        """The CLI header line."""
        sizes = ", ".join(str(len(c)) for c in self.groupset.columns)
        return "Strata = {} (biosamples per stratum: {})".format(len(self), sizes)

    def layout(self, group_cols, comparison, cols, file, null_mode=None):
        """The StrataLayout of one comparison whose groups are the column lists `group_cols` of a matrix of `cols`
        columns (`file`); raises ValueError naming the file for the load-time rules, in their order."""
        gs = self.groupset
        for name, c in zip(gs.names, gs.columns):
            if len(c) and c[-1] >= cols:
                raise ValueError("[--strata] {}: stratum '{}' uses biosample {}, but {} has {} biosamples".format(
                    self.path, name, int(c[-1]) + 1, file, cols))
        stratum_of = np.full(cols, -1, dtype=np.int64)
        for h, c in enumerate(gs.columns):
            stratum_of[c] = h
        group_cols = [np.asarray(c, dtype=np.int64) for c in group_cols]
        compared = np.concatenate(group_cols)
        missing = compared[stratum_of[compared] < 0]
        if len(missing):
            raise ValueError("[--strata] {}: biosample {} of the comparison {} is in no stratum".format(
                self.path, int(missing[0]) + 1, comparison))
        held = [h for h in range(len(gs)) if np.any(stratum_of[compared] == h)]
        sizes = [[int(np.count_nonzero(stratum_of[c] == h)) for c in group_cols] for h in held]
        if not any(sum(1 for n in row if n > 0) >= 2 for row in sizes):
            raise ValueError("[--strata] {}: no stratum holds biosamples of two groups of the comparison {}, so no "
                             "shuffle can move a label".format(self.path, comparison))
        if null_mode == "reference":
            raise ValueError("[--strata] {}: EPILOGOS_B200_NULL=reference replays the reference's unstratified shuffle; "
                             "stratified nulls are drawn on the device".format(self.path))
        return StrataLayout([gs.names[h] for h in held], sizes,
                            [np.concatenate([c[stratum_of[c] == h] for c in group_cols]) for h in held],
                            [np.flatnonzero(stratum_of[compared] == h) for h in held])


class StrataLayout:
    """The strata of one comparison that hold at least one compared biosample, in file order:
      sizes      [H][G] n[h][g], group g's biosamples in stratum h (a biosample of two groups counts in both);
      columns    [H] the matrix columns of stratum h's row, group after group (such a biosample listed twice);
      positions  [H] the same biosamples as ascending positions in the compared matrix, whose columns are the groups'
                 one group after the other (the region null's splits);
      counts     int16 [H, rows, K], each stratum's counts over the shard's rows (set by stratify)."""

    def __init__(self, names, sizes, columns, positions):
        self.names, self.sizes, self.columns, self.positions = names, sizes, columns, positions
        self.counts = None
        self.key = tuple((n, tuple(int(v) for v in c)) for n, c in zip(names, columns))


def parseStrata(path):
    """The Strata of a --strata file (the group-file format); raises GroupFileError with the message of the first
    problem: those of parseGroups naming [--strata], then two strata sharing a biosample."""
    gs = parseGroups(path, flag="--strata")
    for i in range(len(gs)):
        for j in range(i + 1, len(gs)):
            shared = np.intersect1d(gs.columns[i], gs.columns[j])
            if len(shared):
                raise GroupFileError("ERROR: [--strata] strata '{}' and '{}' share biosample {}".format(
                    gs.names[i], gs.names[j], int(shared[0]) + 1))
    return Strata(gs, path)


def stratify(view, strata, null_mode=None):
    """The StrataLayout of the comparison of a paired shard (-a/-b: columns numbered over [A | B]) or of a group view
    (--compare, --multigroup: the numbering of the -i matrix), with its per-stratum counts: one epi_group_counts pass
    over the shard's device matrix, kept with the shard's counts."""
    base = getattr(view, "_shard", view)             # the session.Shard whose device matrix holds the columns
    sel = getattr(view, "selection", None)
    if sel is None:
        c1 = view.states_a.shape[1]
        group_cols, comparison = [np.arange(c1), c1 + np.arange(view.states_b.shape[1])], "[-a] vs [-b]"
    else:
        gs = sel.groupset
        names = list(sel.multi) if sel.multi is not None else [sel.a, sel.b]
        group_cols = [gs.columns[gs.index[n]] for n in names]
        comparison = ",".join(names) if sel.multi is not None else "{}:{}".format(sel.a, sel.b)
    lay = strata.layout(group_cols, comparison, base.width, base.file, null_mode)
    key = ("strata", lay.key)
    if key not in base._counts:
        base._counts[key] = base.backend.stratum_counts(base.states_device(), base.width, base.num_states, lay.columns)
    lay.counts = base._counts[key]
    return lay
