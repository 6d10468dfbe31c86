"""Column-group kernels on the GPU (csrc/groups.cu): epi_group_counts against epi_bin_counts of gathered columns and
against numpy, epi_gather_columns against numpy, and `--groups` runs of the command line against runs on column-subset
files on the same GPU."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import epilogos_oracle as orc
from test_groups import (COLUMNS, GroupBackend, assert_same_outputs, cli, make_inputs, subset_dir)  # noqa: F401

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from epilogos_b200 import engine
    return engine


def group_lists(cols, many, rng):
    """G = 1 (all columns) or G = 64: disjoint ranges, overlapping ranges, scattered subsets, single columns, all."""
    if not many:
        return [np.arange(cols)]
    out = [np.arange(cols)]
    for i in range(8):                                                          # disjoint
        out.append(np.arange(i * cols // 8, (i + 1) * cols // 8))
    for i in range(8):                                                          # overlapping
        out.append(np.arange(i * cols // 16, min(cols, i * cols // 16 + cols // 3)))
    while len(out) < 56:                                                        # scattered
        out.append(np.sort(rng.choice(cols, size=int(rng.integers(2, cols)), replace=False)))
    out += [np.array([int(c)]) for c in rng.choice(cols, size=7, replace=False)] + [np.array([cols - 1])]
    return [g for g in out if len(g)][:64]


def numpy_counts(x, groups, k):
    return np.stack([orc.bin_counts(x[:, g], k) for g in groups]).astype(np.uint16)


@pytest.mark.parametrize("k", [15, 18, 25])
@pytest.mark.parametrize("cols", [127, 833, 2100])
@pytest.mark.parametrize("bins", [77, 1000])
@pytest.mark.parametrize("many", [False, True])
def test_group_counts_equal_gathered_bin_counts_and_numpy(eng, k, cols, bins, many):
    rng = np.random.default_rng(k * 10007 + cols + bins + many)
    x = rng.integers(0, k, size=(bins, cols), dtype=np.int8)
    x[: bins // 5] = k - 1                                                      # long runs of one state
    groups = group_lists(cols, many, rng)
    xd = eng.pack_states(x).cuda()
    got = eng.group_counts(xd, cols, k, groups)
    assert got.shape == (len(groups), bins, k)
    want = numpy_counts(x, groups, k)
    assert np.array_equal(got.cpu().numpy().view(np.uint16), want)
    for g, cols_g in enumerate(groups):
        sub = eng.gather_columns(xd, cols, cols_g)
        assert torch.equal(got[g], eng.bin_counts(sub, len(cols_g), k))
    torch.cuda.synchronize()


@pytest.mark.parametrize("k, cols", [(18, 833), (25, 127)])
def test_group_counts_with_unaligned_pitch_and_base(eng, k, cols):
    from epilogos_b200 import _lib
    rng = np.random.default_rng(5)
    bins, pitch, lead = 300, cols + 5, 3
    x = rng.integers(0, k, size=(bins, cols), dtype=np.int8)
    buf = torch.zeros(lead + bins * pitch, dtype=torch.int8)
    buf[lead:].view(bins, pitch)[:, :cols] = torch.from_numpy(x)
    buf = buf.cuda()
    groups = group_lists(cols, True, rng)[:20]
    flat = torch.from_numpy(np.concatenate(groups).astype(np.int32)).cuda()
    offs = torch.from_numpy(np.concatenate(([0], np.cumsum([len(g) for g in groups]))).astype(np.int32)).cuda()
    out = torch.empty((len(groups), bins, k), dtype=torch.int16, device="cuda")
    _lib.call("epi_group_counts", ctypes.c_void_p(buf.data_ptr() + lead), bins, cols, pitch, k,
              ctypes.c_void_p(flat.data_ptr()), ctypes.c_void_p(offs.data_ptr()), len(groups),
              ctypes.c_void_p(out.data_ptr()), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert np.array_equal(out.cpu().numpy().view(np.uint16), numpy_counts(x, groups, k))


def test_group_counts_reject_bad_lists(eng):
    from epilogos_b200 import _lib
    xd = eng.pack_states(np.zeros((10, 20), dtype=np.int8)).cuda()
    with pytest.raises(_lib.EpilogosB200Error, match="out of range"):
        eng.group_counts(xd, 20, 18, [np.array([3, 20])])
    with pytest.raises(_lib.EpilogosB200Error, match="empty"):
        eng.group_counts(xd, 20, 18, [np.array([1]), np.array([], dtype=np.int32)])
    with pytest.raises(_lib.EpilogosB200Error, match="groups=65"):
        eng.group_counts(xd, 20, 18, [np.array([1])] * 65)


@pytest.mark.parametrize("cols", [20, 833, 2100])
def test_gather_columns_equal_numpy(eng, cols):
    rng = np.random.default_rng(cols)
    x = rng.integers(0, 30, size=(333, cols), dtype=np.int8)
    xd = eng.pack_states(x).cuda()
    for idx in (np.arange(cols), np.array([cols - 1, 0, 5]), np.sort(rng.choice(cols, size=cols // 3, replace=False))):
        got = eng.gather_columns(xd, cols, idx).cpu().numpy()
        assert got.shape == (333, eng.pitch_for(len(idx)))
        assert np.array_equal(got[:, :len(idx)], x[:, idx]) and not got[:, len(idx):].any()


# ---- the command line on the GPU -------------------------------------------------------------------------------------------

SINGLE_GROUPS = ["a", "b", "c", "all", "u"]


@pytest.mark.parametrize("saliency", [1, 2, 3])
def test_single_groups_on_the_gpu_equal_runs_on_subset_files(eng, tmp_path, monkeypatch, saliency):
    from epilogos_b200.backend import CudaBackend
    inp, gfile, meta, data = make_inputs(tmp_path)
    gfile.write_text("".join("%s\t%s\n" % (n, ",".join(str(c + 1) for c in COLUMNS[n])) for n in SINGLE_GROUPS))
    out = tmp_path / "out"
    cli(monkeypatch, CudaBackend(), "-i", inp, "-o", out, "-j", meta, "-s", saliency, "-w", 9, "--groups", gfile)
    for name in SINGLE_GROUPS:
        want = tmp_path / "want" / name
        cli(monkeypatch, CudaBackend(), "-i", subset_dir(tmp_path, data, name), "-o", want, "-j", meta, "-s", saliency,
            "-w", 9)
        assert_same_outputs(out / name, want)


@pytest.mark.parametrize("saliency", [1, 2])
def test_paired_groups_on_the_gpu_equal_two_directory_runs(eng, tmp_path, monkeypatch, saliency):
    from epilogos_b200.backend import CudaBackend
    monkeypatch.setenv("EPILOGOS_B200_SEED", "99")
    inp, gfile, meta, data = make_inputs(tmp_path)
    common = ["-j", meta, "-s", saliency, "-w", 9, "-n", "-t", 5, "-z", 150]
    out = tmp_path / "out"
    cli(monkeypatch, CudaBackend(), "-m", "paired", "-i", inp, "-o", out, "--groups", gfile, "--compare", "a:b",
        "--compare", "c:u", *common)
    for a, b in (("a", "b"), ("c", "u")):
        want = tmp_path / "want" / ("%s_vs_%s" % (a, b))
        cli(monkeypatch, CudaBackend(), "-m", "paired", "-a", subset_dir(tmp_path, data, a), "-b",
            subset_dir(tmp_path, data, b), "-o", want, *common)
        assert_same_outputs(out / want.name, want)
