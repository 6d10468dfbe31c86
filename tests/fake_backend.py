"""Stand-in compute provider for CPU-only tests of the HOST logic (sharding, all-reduce, gather, file naming).
It answers the backend interface of epilogos_b200/backend.py with the oracle.  Test infrastructure only: the
product never imports this, and epilogos_b200 itself has no CPU path."""
import numpy as np
import torch

import sampler_oracle as so
from oracle import epilogos_oracle as orc


class OracleBackend:
    name = "oracle-test-double"

    def counts(self, states0, num_states):
        return torch.from_numpy(orc.bin_counts(states0, num_states).astype(np.uint16).view(np.int16))

    @staticmethod
    def _cnt(cnt):
        return cnt.numpy().view(np.uint16).astype(np.int64)

    def add_counts(self, cnt_a, cnt_b):
        return cnt_a + cnt_b

    def expected_table(self, cnt, width, saliency):
        c = self._cnt(cnt)
        if saliency == 1:
            return torch.from_numpy(c.sum(axis=0))
        n2 = c.T @ c
        n2[np.diag_indices(c.shape[1])] -= c.sum(axis=0)
        return torch.from_numpy(n2)

    def normalize(self, counts):
        return torch.from_numpy(orc.normalize_expected(counts.numpy()))

    def to_device(self, array):
        return torch.as_tensor(array)

    def scores(self, cnt, width, saliency, exp, perms=None, exact=False):
        c = self._cnt(cnt)
        if saliency == 1:
            return torch.from_numpy(orc.s1_scores_from_counts(c, width, exp.numpy()))
        return torch.from_numpy(orc.s2_scores_from_counts(c, perms or width * (width - 1), exp.numpy()))

    # paired mode
    def shuffled_counts_perm(self, states_a, states_b, perm, num_states, size_a, size_b):
        gs = -1 if (size_a, size_b) == (states_a.shape[1], states_b.shape[1]) else size_a
        sa, sb = orc.paired_split(states_a, states_b, perm, gs)
        return self.counts(sa, num_states), self.counts(sb, num_states)

    def shuffled_counts_device(self, cnt_a, cnt_b, size_a, size_b, seed, nperm=1, width=None, bin_offset=0):
        """The device's draws (sampler_oracle.draw_shuffle): permutation p of row r from the stream keyed by (seed, p,
        GLOBAL bin bin_offset + r)."""
        a, b = self._cnt(cnt_a), self._cnt(cnt_b)
        rows, k = a.shape
        r = so.draw_shuffle(seed, np.repeat(np.arange(nperm), rows), bin_offset + np.tile(np.arange(rows), nperm),
                            np.tile(a, (nperm, 1)), np.tile(b, (nperm, 1)), size_a, size_b)
        ta = torch.from_numpy(r["a"].reshape(nperm, rows, k).astype(np.uint16).view(np.int16))
        tb = torch.from_numpy(r["b"].reshape(nperm, rows, k).astype(np.uint16).view(np.int16))
        return (ta[0], tb[0]) if nperm == 1 else (ta, tb)

    def pairwise_combine(self, score_a, score_b, null_a, null_b):
        delta = None if score_a is None else score_a - score_b
        dist = None
        if null_a is not None:
            d = (null_a - null_b).numpy()
            dist = torch.from_numpy(np.sum(np.square(d), axis=1) * np.sign(np.sum(d, axis=1)))
        return delta, dist

    def quiescent_mask(self, cnt_a, cols_a, cnt_b, cols_b, q):
        a, b = self._cnt(cnt_a), self._cnt(cnt_b)
        if q == -1:
            return torch.zeros(a.shape[0], dtype=torch.uint8)
        return torch.from_numpy(((a[:, q] == cols_a) & (b[:, q] == cols_b)).astype(np.uint8))
