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

    def group_counts(self, x_dev, cols, num_states, groups):
        """Counts of every column group (lists of 0-based columns) of a device matrix, one pass: a list of [rows, K]
        blocks.  The count kernels' consumers need 16-byte aligned counts, so a block that does not start on 16 bytes
        (rows * K * 2 not a multiple of 16) is copied."""
        with timing.stage("kernels", sync_cuda=True):
            cnt = engine.group_counts(x_dev, cols, num_states, groups)
        return [c if c.data_ptr() % 16 == 0 else c.clone() for c in cnt]

    def gather_columns(self, x_dev, cols, idx):
        """The matrix of the columns idx of a device matrix, on the device."""
        return engine.gather_columns(x_dev, cols, idx)

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
        on_device = getattr(states0, "device_matrix", None)      # a group's columns, gathered on the device (groups.py)
        return on_device() if on_device is not None else self._upload(states0)

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

    def permutation_exceedances(self, cnt_a, cnt_b, dist, nperm, seed, size_a, size_b, width, bin_offset, saliency, exp,
                                score_widths, perms, exact=False, workspace_bytes=1 << 30):
        """Per-bin permutation counts k[b] = #{p < nperm : |null(b, p)| >= |dist[b]|} (int32 tensor holding uint32): the
        null distances of permutations 0 .. nperm-1 drawn as shuffled_counts_device draws them, A' scored at
        score_widths[0] with perms[0], B' at score_widths[1] with perms[1], in the run's score mode (`exact`).
        S1 runs the fused kernel (its TABLE and DIRECT values are the same numbers); S2 and tables wider than the S1
        value table loop over bin chunks x permutation blocks of draw + score + count, whose device buffers stay below
        `workspace_bytes`.  The result does not depend on that cap."""
        rows, k_states = cnt_a.shape
        exp = exp.to(self.device).contiguous()
        dist = dist.to(self.device).contiguous()
        k = torch.zeros(rows, dtype=torch.int32, device=self.device)
        if saliency == 1 and max(score_widths) <= engine.S1_TABLE_MAX_WIDTH:
            with timing.stage("kernels", sync_cuda=True):
                return engine.permutation_exceedances_s1(cnt_a, cnt_b, size_a, size_b, seed, 0, nperm, width, bin_offset,
                                                         exp, score_widths[0], score_widths[1], dist, k)
        with timing.stage("kernels", sync_cuda=True):
            # A', B' counts (uint16) and scores (float32)
            for lo, hi, p0, n in self._blocks(rows, nperm, workspace_bytes, 12 * k_states):
                oa, ob = engine.shuffled_counts_philox_range(cnt_a[lo:hi], cnt_b[lo:hi], size_a, size_b, seed, p0, n,
                                                             width, bin_offset=bin_offset + lo)
                sa = self.scores(oa.reshape(-1, k_states), score_widths[0], saliency, exp, perms=perms[0], exact=exact)
                sb = self.scores(ob.reshape(-1, k_states), score_widths[1], saliency, exp, perms=perms[1], exact=exact)
                engine.null_exceedances(sa.reshape(n, hi - lo, k_states), sb.reshape(n, hi - lo, k_states),
                                        dist[lo:hi], k[lo:hi])
        return k

    # -- multi-group comparisons ------------------------------------------------------------------------
    def _group_scores(self, cnt, n, saliency, exp, exact, out=None):
        """Scores of one group's counts [bins, K] at its own width n (S2 over its n (n - 1) ordered pairs), into `out`
        when given.  The score kernels want 16-byte aligned counts and outputs; the callers keep their blocks aligned
        except for a tail of fewer than 8 bins, whose blocks are copied."""
        cnt = cnt if cnt.data_ptr() % 16 == 0 else cnt.clone()
        direct = out is not None and out.data_ptr() % 16 != 0
        o32 = None if out is None or direct else out
        if saliency == 1:
            sc = engine.scores_s1(cnt, n, exp, out32=o32)
        else:
            sc = engine.scores_s2(cnt, n, exp, perms=n * (n - 1), out32=o32,
                                  mode=engine.EPI_SCORE_DIRECT if exact else engine.EPI_SCORE_TABLE)
        if direct:
            out.copy_(sc)
        return sc if out is None else out

    @staticmethod
    def _blocks(rows, nperm, workspace_bytes, cell_bytes):
        """(lo, hi, p0, n): bin chunks [lo, hi) x permutation blocks p0 .. p0 + n - 1 whose buffers, `cell_bytes` per
        (bin, shuffle), stay below `workspace_bytes` (eight bins and one shuffle at the least).  Chunk lengths are
        multiples of 8, then comes the tail of rows % 8 bins: every [.., hi - lo, K] block of uint16 counts or float32
        scores then starts on 16 bytes, except in the tail."""
        cells = max(1, int(workspace_bytes) // cell_bytes)
        body = rows - rows % 8
        step = max(8, cells - cells % 8)
        edges = list(range(0, body, step)) + [body]
        for lo, hi in list(zip(edges[:-1], edges[1:])) + ([(body, rows)] if body < rows else []):
            block = max(1, min(nperm, cells // (hi - lo)))
            for p0 in range(0, nperm, block):
                yield lo, hi, p0, min(block, nperm - p0)

    def multigroup_stat(self, cnt, sizes, saliency, exp, exact=False, workspace_bytes=1 << 30):
        """(T float64, g* uint8, s* uint8, sign int8), each [bins], of the groups' counts cnt int16 [G, bins, K] (group g
        of width sizes[g]) scored against exp in the run's score mode (`exact`).  Bins go in chunks whose G score arrays
        stay below `workspace_bytes`."""
        G, rows, k_states = cnt.shape
        exp = exp.to(self.device).contiguous()
        out = (torch.empty(rows, dtype=torch.float64, device=self.device),
               torch.empty(rows, dtype=torch.uint8, device=self.device),
               torch.empty(rows, dtype=torch.uint8, device=self.device),
               torch.empty(rows, dtype=torch.int8, device=self.device))
        with timing.stage("kernels", sync_cuda=True):
            # bin chunks only: with one "shuffle" every chunk is a single block
            for lo, hi, _, _ in self._blocks(rows, 1, workspace_bytes, 4 * G * k_states):
                sc = torch.empty((G, hi - lo, k_states), dtype=torch.float32, device=self.device)
                for g, n in enumerate(sizes):
                    self._group_scores(cnt[g, lo:hi], n, saliency, exp, exact, out=sc[g])
                for dst, src in zip(out, engine.multigroup_stat(sc, sizes)):
                    dst[lo:hi] = src
        return out

    def multigroup_exceedances(self, cnt, sizes, t, nperm, seed, bin_offset, saliency, exp, exact=False,
                               workspace_bytes=1 << 30):
        """Per-bin permutation counts k[b] = #{p < nperm : T_null(b, p) >= t[b]} (int32 tensor holding uint32) of the
        groups' counts cnt int16 [G, bins, K]: shuffle p drawn as engine.multigroup_shuffled_counts_range draws it, group
        g scored at width sizes[g] in the run's score mode.  S1 runs the fused kernel where its tables fit; S2 and wider
        S1 groups loop over bin chunks x permutation blocks of draw + score + count, whose device buffers (shuffled
        counts and their scores) stay below `workspace_bytes`.  The result does not depend on that cap."""
        G, rows, k_states = cnt.shape
        exp = exp.to(self.device).contiguous()
        t = t.to(self.device).contiguous()
        k = torch.zeros(rows, dtype=torch.int32, device=self.device)
        if saliency == 1 and engine.multigroup_s1_fused_fits(sizes, k_states):
            with timing.stage("kernels", sync_cuda=True):
                return engine.multigroup_exceedances_s1(cnt, sizes, seed, 0, nperm, bin_offset, exp, t, k)
        with timing.stage("kernels", sync_cuda=True):
            # shuffled counts (uint16) and scores (float32)
            for lo, hi, p0, n in self._blocks(rows, nperm, workspace_bytes, 6 * G * k_states):
                oc = engine.multigroup_shuffled_counts_range(cnt[:, lo:hi], sizes, seed, p0, n, bin_offset + lo)
                sc = torch.empty((n, G, hi - lo, k_states), dtype=torch.float32, device=self.device)
                for p in range(n):
                    for g, size in enumerate(sizes):
                        self._group_scores(oc[p, g], size, saliency, exp, exact, out=sc[p, g])
                del oc
                engine.multigroup_null_exceedances(sc, sizes, t[lo:hi], k[lo:hi])
        return k

    # -- region null: whole-genome label permutations (epilogos_b200.region_null) ------------------------------------
    def region_maxima_paired(self, x_dev, halo, sizes, num_states, window, nperm, seed, saliency, exp, exact=False,
                             workspace_bytes=1 << 30):
        """int64 [nperm] on the device: for split p of region_null.split_blocks, the largest sum of W = `window`
        consecutive q(|distance|) of the rows of x_dev (the [A | B] label matrix, A of sizes[0] columns) followed by the
        host rows `halo`.  Each permuted group is scored like its real counterpart (its width, S2 normaliser and score
        mode) and reduced with the text round trip, so the identity split gives the real distances.  -1 where no window
        fits."""
        def stat(cnt, n0, out):
            sa = self._group_scores(cnt[0], sizes[0], saliency, exp, exact)
            sb = self._group_scores(cnt[1], sizes[1], saliency, exp, exact)
            delta, _ = engine.pairwise_combine(sa, sb)
            d, _ = engine.pairwise_real_reduce(delta, True)
            torch.abs(d, out=out)
        return self._region_maxima(x_dev, halo, sizes, num_states, window, nperm, seed, exp, torch.float32,
                                   12 * num_states + 16, stat, workspace_bytes)

    def region_maxima_multigroup(self, x_dev, halo, sizes, num_states, window, nperm, seed, saliency, exp, exact=False,
                                 workspace_bytes=1 << 30):
        """As region_maxima_paired for the multi-group statistic T of the groups, which are the consecutive column slices
        of sizes[0], sizes[1], ... of x_dev."""
        G = len(sizes)

        def stat(cnt, n0, out):
            sc = torch.empty((G, n0, num_states), dtype=torch.float32, device=self.device)
            for g, n in enumerate(sizes):
                self._group_scores(cnt[g], n, saliency, exp, exact, out=sc[g])
            out.copy_(engine.multigroup_stat(sc, sizes)[0])
        return self._region_maxima(x_dev, halo, sizes, num_states, window, nperm, seed, exp, torch.float64,
                                   6 * G * num_states + 16, stat, workspace_bytes)

    def _region_maxima(self, x_dev, halo, sizes, num_states, window, nperm, seed, exp, dtype, cell_bytes, stat,
                       workspace_bytes):
        """Split blocks (drawn in order, outer) x bin chunks (inner, overlapping by W - 1 rows): split counts, the
        statistic of every split into one [splits, rows] array, its windowed maxima.  Buffers stay near
        `workspace_bytes`; the result does not depend on it."""
        from . import region_null
        exp = exp.to(self.device).contiguous()
        N, G = int(sum(sizes)), len(sizes)
        x = x_dev
        if halo is not None and len(halo):
            h = np.zeros((len(halo), x_dev.shape[1]), dtype=np.int8)
            h[:, :N] = halo
            x = torch.cat([x_dev, torch.from_numpy(h).to(self.device)])
        rows = x.shape[0]
        maxima = torch.full((nperm,), -1, dtype=torch.int64, device=self.device)
        starts = rows - window + 1
        if starts <= 0:
            return maxima
        cells = max(1, int(workspace_bytes) // cell_bytes)
        # long chunks, and as many splits per block as fit: the bitsets of a tile are built once per launch
        chunk = min(starts, max(1 << 16, cells // nperm))
        block = max(1, min(nperm, cells // (chunk + window - 1)))
        with timing.stage("kernels", sync_cuda=True):
            for p0, members in region_null.split_blocks(seed, sizes, nperm, block):
                n = members.shape[0]
                mem = torch.from_numpy(members.view(np.int64)).to(self.device)
                for lo in range(0, starts, chunk):
                    hi = min(rows, lo + chunk + window - 1)
                    cnt = engine.split_counts(x[lo:hi], N, num_states, mem, G)
                    vals = torch.empty((n, hi - lo), dtype=dtype, device=self.device)
                    for p in range(n):
                        stat(cnt[p], hi - lo, vals[p])
                    del cnt
                    engine.window_max(vals, window, maxima[p0:p0 + n])
        return maxima

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
