"""ChromHMM state-by-line files -> input matrices (epilogos_b200.preprocess, the native form of the reference's
bin/preprocess_data_ChromHMM.sh): byte-identical `matrix_<chr>.txt` files and messages, against a restatement of the
script's paste / awk recipe everywhere and against the UNMODIFIED script and its example data where EPILOGOS_REFERENCE names a
checkout of the reference."""
import gzip
import io
import subprocess
from pathlib import Path

import numpy as np
import pytest

from epilogos_b200 import helpers, preprocess
from epilogos_b200._lib import EpilogosB200Error
from oracle import stage_reference

REFERENCE = stage_reference.SOURCE if stage_reference.source_available() else None
SCRIPT = REFERENCE / "bin" / "preprocess_data_ChromHMM.sh" if REFERENCE else None
EXAMPLE = REFERENCE / "data" / "ChromHMM" if REFERENCE else None


def _statebyline(path, biosample, chrom, labels, gz):
    text = "%s\t%s\nMaxState E\n%s\n" % (biosample, chrom, "\n".join(str(int(v)) for v in labels))
    if gz:
        with gzip.open(path, "wt") as f:
            f.write(text)
    else:
        Path(path).write_text(text)


def _paste_awk(columns, chrom):
    """preprocess_data_ChromHMM.sh:46-49 restated: rows of the pasted label columns behind `chr, (NR-3)*200, (NR-2)*200`."""
    rows = len(columns[0])
    return "".join("%s\t%d\t%d\t%s\n" % (chrom, r * 200, (r + 1) * 200, "\t".join(str(int(c[r])) for c in columns))
                   for r in range(rows))


def _synthetic(tmp_path, rng):
    data = tmp_path / "calls"
    data.mkdir()
    samples = ["BSS%05d" % i for i in (7, 3, 11, 5)]                # metadata order, not alphabetical
    (tmp_path / "meta.tsv").write_text("id\tother\n" + "".join("%s\tx\n" % s for s in samples + ["BSS99999"]))
    (tmp_path / "sizes.genome").write_text("chr1\t1000\nchr2\t800\nchrX\t500\n")
    cols = {}
    for chrom, bins in (("chr1", 317), ("chrX", 41)):
        for j, s in enumerate(samples):
            if chrom == "chrX" and s == "BSS00011":
                continue                                            # a biosample without this chromosome is skipped
            labels = rng.integers(1, 26, bins)
            labels[rng.random(bins) < 0.4] = 25
            cols.setdefault(chrom, []).append(labels)
            _statebyline(data / ("%s_25_CALLS_PER_LINE_%s_statebyline.txt%s" % (s, chrom, ".gz" if j % 2 else "")), s, chrom,
                         labels, gz=bool(j % 2))
    return data, cols


def test_matrices_equal_the_scripts_recipe(tmp_path):
    rng = np.random.default_rng(41)
    data, cols = _synthetic(tmp_path, rng)
    log = io.StringIO()
    written = preprocess.main(data, tmp_path / "meta.tsv", tmp_path / "sizes.genome", tmp_path / "out", out=log)
    assert log.getvalue() == ("Processing chr1: 4 files found. Done.\nProcessing chr2: 0 files found. Skipping.\n"
                              "Processing chrX: 3 files found. Done.\n")
    assert [p.name for p in written] == ["matrix_chr1.txt", "matrix_chrX.txt"]
    for chrom in ("chr1", "chrX"):
        assert (tmp_path / "out" / ("matrix_%s.txt" % chrom)).read_text() == _paste_awk(cols[chrom], chrom)
    # gzipped output holds the same text and goes straight into the matrix reader
    preprocess.main(data, tmp_path / "meta.tsv", tmp_path / "sizes.genome", tmp_path / "outz", gzip_level=4, out=io.StringIO())
    with gzip.open(tmp_path / "outz" / "matrix_chr1.txt.gz", "rt") as f:
        assert f.read() == _paste_awk(cols["chr1"], "chr1")
    loc, m = helpers.read_matrix(tmp_path / "outz" / "matrix_chr1.txt.gz", num_states=25)
    assert np.array_equal(m, np.stack(cols["chr1"], axis=1) - 1) and loc["chrom"][0] == "chr1" and loc["end"][-1] == 317 * 200
    # the matrix without any text in between
    files = preprocess.find_files(data, preprocess.biosamples(tmp_path / "meta.tsv"), "chr1")
    direct, chrom = preprocess.read_chromosome(files, num_states=25)
    assert chrom == "chr1" and direct.dtype == np.int8 and np.array_equal(direct, m)
    if SCRIPT and SCRIPT.is_file():                                 # the unmodified script on the same files
        ref = tmp_path / "ref"
        ref.mkdir()
        r = subprocess.run(["bash", str(SCRIPT), str(data), str(tmp_path / "meta.tsv"), str(tmp_path / "sizes.genome")], cwd=ref,
                           capture_output=True, text=True)
        assert r.returncode == 0 and r.stdout == log.getvalue()
        for chrom in ("chr1", "chrX"):
            assert (ref / ("matrix_%s.txt" % chrom)).read_bytes() == (tmp_path / "out" / ("matrix_%s.txt" % chrom)).read_bytes()


def test_more_biosamples_than_one_column_group(tmp_path):
    """Columns are parsed contiguously and turned into rows in groups of 256: 300 biosamples cross a group boundary."""
    rng = np.random.default_rng(43)
    data = tmp_path / "calls"
    data.mkdir()
    n, bins = 300, 53
    x = rng.integers(1, 16, size=(bins, n))
    (tmp_path / "meta.tsv").write_text("id\n" + "".join("S%04d\n" % j for j in range(n)))
    (tmp_path / "sizes.genome").write_text("chr21\t48129895\n")
    for j in range(n):
        _statebyline(data / ("S%04d_15_chr21_statebyline.txt" % j), "S%04d" % j, "chr21", x[:, j], gz=False)
    files = preprocess.find_files(data, preprocess.biosamples(tmp_path / "meta.tsv"), "chr21")
    m, chrom = preprocess.read_chromosome(files, num_states=15)
    assert chrom == "chr21" and np.array_equal(m, x - 1) and not m.base[:, n:].any()
    preprocess.main(data, tmp_path / "meta.tsv", tmp_path / "sizes.genome", tmp_path / "out", out=io.StringIO())
    assert (tmp_path / "out" / "matrix_chr21.txt").read_text() == _paste_awk([x[:, j] for j in range(n)], "chr21")


def test_bad_inputs_are_errors(tmp_path):
    data = tmp_path / "calls"
    data.mkdir()
    (tmp_path / "meta.tsv").write_text("id\nA1\nB2\n")
    (tmp_path / "sizes.genome").write_text("chr1\t1000\n")
    _statebyline(data / "A1_chr1_statebyline.txt", "A1", "chr1", [1, 2, 3, 4], gz=False)
    _statebyline(data / "B2_chr1_statebyline.txt", "B2", "chr1", [1, 2, 3], gz=False)
    with pytest.raises(ValueError, match="holds 3 bins"):           # paste would pad the short file with empty fields
        preprocess.main(data, tmp_path / "meta.tsv", tmp_path / "sizes.genome", tmp_path / "out", out=io.StringIO())
    _statebyline(data / "B2_chr1_statebyline.txt", "B2", "chr1", [1, 2, 19, 4], gz=False)
    with pytest.raises(EpilogosB200Error, match="line 5: state 19 outside 1..18"):
        preprocess.main(data, tmp_path / "meta.tsv", tmp_path / "sizes.genome", tmp_path / "out", num_states=18, out=io.StringIO())
    (data / "B2_chr1_statebyline.txt").write_text("B2\tchr1\nMaxState E\n1\nx\n")
    with pytest.raises(EpilogosB200Error, match="not an integer"):
        preprocess.main(data, tmp_path / "meta.tsv", tmp_path / "sizes.genome", tmp_path / "out", out=io.StringIO())
    _statebyline(data / "B2_chr1_statebyline.txt", "B2", "chr1", [1, 2, 3, 4], gz=False)
    _statebyline(data / "B2_rep2_chr1_statebyline.txt", "B2", "chr1", [1, 2, 3, 4], gz=False)
    with pytest.raises(ValueError, match="more than one file"):
        preprocess.main(data, tmp_path / "meta.tsv", tmp_path / "sizes.genome", tmp_path / "out", out=io.StringIO())


def test_matrix_writer_matches_python_formatting(tmp_path):
    """epi_write_matrix_tsv: one-, two- and three-digit labels, many rows (several writer blocks), plain and gzip."""
    rng = np.random.default_rng(42)
    x = rng.integers(0, 127, size=(9000, 37)).astype(np.int8)
    x[:, 0] = 126
    want = "".join("chr7_random\t%d\t%d\t%s\n" % (r * 200, (r + 1) * 200, "\t".join(str(int(v) + 1) for v in x[r])) for r in range(len(x)))
    preprocess.write_matrix(tmp_path / "m.txt", "chr7_random", x)
    assert (tmp_path / "m.txt").read_text() == want
    preprocess.write_matrix(tmp_path / "m.txt.gz", "chr7_random", x, gzip_level=1, threads=3)
    with gzip.open(tmp_path / "m.txt.gz", "rt") as f:
        assert f.read() == want
    assert np.array_equal(helpers.read_matrix(tmp_path / "m.txt.gz", num_states=127)[1], x)
    preprocess.write_matrix(tmp_path / "e.txt.gz", "chr1", np.zeros((0, 5), np.int8), gzip_level=6)
    with gzip.open(tmp_path / "e.txt.gz", "rb") as f:
        assert f.read() == b""


@pytest.mark.skipif(not (SCRIPT and SCRIPT.is_file() and EXAMPLE.is_dir()),
                    reason="needs the reference's script and example data (EPILOGOS_REFERENCE)")
def test_real_example_data_against_the_unmodified_script(tmp_path, golden):
    """The reference's own example (10 biosamples, chr1, 1,246,253 bins): the script's matrix_chr1.txt byte for byte, and the
    matrix read directly from the state-by-line files equals the matrix the goldens were generated from."""
    (tmp_path / "sizes.genome").write_text("chr1\t249250621\nchr2\t243199373\n")
    meta = REFERENCE / "data" / "metadata_Boix.txt"
    ref = tmp_path / "ref"
    ref.mkdir()
    r = subprocess.run(["bash", str(SCRIPT), str(EXAMPLE), str(meta), str(tmp_path / "sizes.genome")], cwd=ref, capture_output=True,
                       text=True)
    assert r.returncode == 0
    log = io.StringIO()
    preprocess.main(EXAMPLE, meta, tmp_path / "sizes.genome", tmp_path / "out", out=log)
    assert log.getvalue() == r.stdout
    assert (tmp_path / "out" / "matrix_chr1.txt").read_bytes() == (ref / "matrix_chr1.txt").read_bytes()
    files = preprocess.find_files(EXAMPLE, preprocess.biosamples(meta), "chr1")
    direct, chrom = preprocess.read_chromosome(files, num_states=18)
    # the goldens pasted the files in alphabetical order (SURVEY Appendix B); the script takes the metadata's order
    alphabetical = np.argsort([Path(f).name for f in files])
    assert chrom == "chr1" and np.array_equal(direct[:, alphabetical], golden("real10_chr1_full")["x"])
