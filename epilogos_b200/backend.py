"""The compute provider used by the stage drivers.

CudaBackend is the product: every method is a call into libepilogos_b200.so (via engine) on the current
CUDA device, and it raises if the library or a B200 is missing -- there is no CPU fallback.  The stage
drivers take the backend as a parameter only so that the CPU-only unit tests can exercise the
sharding / all-reduce / gather / file-naming logic with a stand-in defined under tests/.
"""
import numpy as np
import torch

from . import engine, timing


class CudaBackend:
    name = "cuda"

    def __init__(self, device=None):
        if not torch.cuda.is_available():
            raise RuntimeError("epilogos_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        engine.device_info()

    # -- per-bin counts of a shard (numpy int8 [rows, C], 0-based) -> device tensor [rows, K] (uint16 in int16)
    def _upload(self, states0):
        """numpy int8 [rows, C] -> device [rows, pitch].  Matrices that come from helpers.read_matrix are views of an
        already pitched (and possibly pinned) buffer and are uploaded as they are."""
        with timing.stage("host -> device", sync_cuda=True):
            return self._upload_impl(states0)

    def _upload_impl(self, states0):
        base = getattr(states0, "base", None)
        if (isinstance(base, np.ndarray) and base.dtype == np.int8 and base.ndim == 2 and base.flags.c_contiguous
                and base.shape[0] == states0.shape[0] and base.shape[1] % 16 == 0 and base.shape[1] >= states0.shape[1]
                and (states0.size == 0 or states0.ctypes.data == base.ctypes.data)):
            return torch.from_numpy(base).to(self.device, non_blocking=True)
        return engine.pack_states(states0).to(self.device, non_blocking=True)

    def counts(self, states0, num_states):
        x = self._upload(states0)
        with timing.stage("kernels", sync_cuda=True):
            return engine.bin_counts(x, states0.shape[1], num_states)

    def add_counts(self, cnt_a, cnt_b):
        """Counts of the concatenated matrix [A | B] (helpers.py:173-179) = sum of the group counts."""
        return (cnt_a + cnt_b).contiguous()

    # -- integer expected table of the shard: int64 [K] (S1) or [K, K] (S2), on the device
    def expected_table(self, cnt, width, saliency):
        with timing.stage("kernels", sync_cuda=True):
            n1, n2 = engine.expected_tables(cnt, width, want_s1=saliency == 1, want_s2=saliency == 2)
        return n1 if saliency == 1 else n2

    def normalize(self, counts):
        return engine.normalize(counts.to(self.device))

    def to_device(self, array):
        return torch.as_tensor(array).to(self.device)

    # -- float32 scores [rows, K] of the shard
    def scores(self, cnt, width, saliency, exp, perms=None, exact=False):
        """`exact`: evaluate the S2 terms one by one with the reference's float64 expression (EPI_SCORE_DIRECT) instead
        of the tensor-core TABLE form; S1 is exact either way (its value table is built with that expression)."""
        exp = exp.to(self.device).contiguous()
        with timing.stage("kernels", sync_cuda=True):
            if saliency == 1:
                return engine.scores_s1(cnt, width, exp)
            return engine.scores_s2(cnt, width, exp, perms=perms,
                                    mode=engine.EPI_SCORE_DIRECT if exact else engine.EPI_SCORE_TABLE)

    # -- S3 ------------------------------------------------------------------------------------------
    def states_to_device(self, states0):
        return self._upload(states0)

    def s3_tiles(self, x_dev, width, num_states):
        """Upper-triangular tiles of the shard's one-hot Gram matrix (int32): the tensor that is all-reduced."""
        return engine.s3_expected_tiles(x_dev, width, num_states)

    def s3_counts(self, tiles, plan, width, num_states, total_bins):
        counts, _ = engine.s3_finalize(tiles, width, num_states, plan["mp"], total_bins, want_counts=True,
                                       want_exp=False)
        return counts

    def scores_s3(self, x_dev, width, num_states, exp):
        terms = engine.s3_terms(exp.to(self.device).contiguous().reshape(-1), width, num_states)
        return engine.scores_s3(x_dev, width, num_states, terms)

    # -- paired mode -----------------------------------------------------------------------------------
    def shuffled_counts_perm(self, states_a, states_b, perm, num_states, size_a, size_b):
        xa, xb = self.states_to_device(states_a), self.states_to_device(states_b)
        p = torch.as_tensor(perm.astype("int32", copy=False)).to(self.device)
        return engine.shuffled_counts_perm(xa, states_a.shape[1], xb, states_b.shape[1], p.contiguous(), num_states,
                                           size_a, size_b)

    def shuffled_counts_device(self, cnt_a, cnt_b, size_a, size_b, seed, nperm=1, width=None, bin_offset=0):
        oa, ob = engine.shuffled_counts_philox(cnt_a, cnt_b, size_a, size_b, seed, nperm, width=width,
                                               bin_offset=bin_offset)
        return (oa[0], ob[0]) if nperm == 1 else (oa, ob)

    def pairwise_combine(self, score_a, score_b, null_a, null_b):
        return engine.pairwise_combine(score_a, score_b, null_a, null_b)

    def quiescent_mask(self, cnt_a, cols_a, cnt_b, cols_b, quiescent_state):
        return engine.quiescent_mask(cnt_a, cols_a, cnt_b, cols_b, quiescent_state)

    def pairwise_real_reduce(self, delta, text_round_trip=True):
        return engine.pairwise_real_reduce(delta.to(self.device).contiguous(), text_round_trip)

    # -- paired statistics (step 4) ---------------------------------------------------------------------
    def null_pool(self, null_dist, quiescent):
        return engine.null_compact(null_dist.to(self.device).contiguous(), quiescent.to(self.device).contiguous())

    def null_subsample(self, pool, trials, size, seed):
        return engine.null_subsample(pool, trials, size, seed)

    def gennorm_fit(self, samples):
        params, status = engine.gennorm_fit(samples)
        return params.cpu().numpy(), status.cpu().numpy()

    def gennorm_pvalues(self, x, beta, loc, scale):
        return engine.gennorm_pvalues(x.to(self.device).contiguous(), beta, loc, scale)

    def bh_adjust(self, p):
        return engine.bh_adjust(p)
