"""CPU-side checks of the C-ABI library: it loads without a GPU and exports every symbol the header declares;
compute entry points fail loudly (no CPU fallback) when there is no device."""
import ctypes
import re
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent


@pytest.fixture(scope="module")
def lib():
    from epilogos_b200 import build, _lib
    build.build()
    return _lib.load()


def header_functions():
    text = (ROOT / "include" / "epilogos_b200.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(epi_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_are_exported(lib):
    names = header_functions()
    assert "epi_bin_counts" in names and "epi_single_host" in names
    for name in names:
        assert hasattr(lib, name), "symbol %s declared in include/epilogos_b200.h is not exported" % name


def test_ctypes_prototypes_cover_header():
    from epilogos_b200 import _lib
    assert sorted(_lib.PROTOTYPES) == header_functions()


def test_abi_version(lib):
    assert lib.epi_abi_version() == 1


def test_no_cpu_fallback(lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from epilogos_b200 import _lib
    with pytest.raises(_lib.EpilogosB200Error):
        _lib.call("epi_bin_counts", ctypes.c_void_p(16), 1, 1, 16, 18, ctypes.c_void_p(16), ctypes.c_void_p(0))
    msg = lib.epi_last_error().decode()
    assert "no CPU fallback" in msg or "CUDA" in msg


@pytest.mark.parametrize("bins,cols,k", [(0, 2, 1), (1, 16, 16), (129, 17, 16), (300_001, 833, 18), (20_001, 1422, 18),
                                         (50_001, 400, 25), (7, 4096, 32)])
def test_s3_plan_closed_form(lib, bins, cols, k):
    """epi_s3_plan (no device needed): one-hot rows padded to 256-row blocks, bins to 128-bin k-steps, the 128 x 256 tiles
    of the blocks on or above the diagonal, and the tile buffer with its (row tile, block column) -> tile index behind.
    C*K = 131,072 is the largest schedule (512 block columns in 64 raster groups)."""
    from epilogos_b200 import engine
    mp = -(-cols * k // 256) * 256
    bp = -(-bins // 128) * 128
    nt = mp // 256
    ntiles = nt * (nt + 1)
    assert engine.s3_plan(bins, cols, k) == dict(mp=mp, bp=bp, ntiles=ntiles, onehot_bytes=mp * bp,
                                                 tile_bytes=ntiles * 128 * 256 * 4 + (mp // 128) * nt * 4)


def test_s3_plan_refuses_a_schedule_past_64_raster_groups(lib):
    from epilogos_b200 import _lib, engine
    assert engine.s3_plan(1, 4096, 32)["mp"] == 131072
    with pytest.raises(_lib.EpilogosB200Error, match="biosamples x states = 131073 is too large for the S3 tile schedule"):
        engine.s3_plan(1, 43691, 3)


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    """No silent fallback: if the shared library is absent the binding raises with build instructions."""
    from epilogos_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", tmp_path / "libepilogos_b200.so")
    with pytest.raises(_lib.EpilogosB200Error, match="no CPU fallback"):
        _lib.call("epi_abi_version")
    with pytest.raises(_lib.EpilogosB200Error):
        from epilogos_b200 import helpers
        helpers.countRows(__file__)


def test_product_never_imports_the_oracle():
    """oracle/ is test infrastructure: nothing under epilogos_b200/ may import it."""
    import re
    pkg = ROOT / "epilogos_b200"
    for f in pkg.rglob("*.py"):
        text = f.read_text()
        assert not re.search(r"^\s*(from|import)\s+oracle\b", text, flags=re.M), f


def test_header_is_plain_c(tmp_path):
    """The drop-in boundary is a C ABI: the header compiles as C99 and as C++11 with warnings as errors (plain pointers and
    sizes only, nothing from torch or CUDA in a signature)."""
    import shutil
    import subprocess
    if shutil.which("gcc") is None or shutil.which("g++") is None:
        pytest.skip("no host compiler")
    for cc, std, name in (("gcc", "-std=c99", "h.c"), ("g++", "-std=c++11", "h.cpp")):
        src = tmp_path / name
        src.write_text('#include "epilogos_b200.h"\nint main(void) { return epi_abi_version() == EPI_ABI_VERSION ? 0 : 1; }\n')
        r = subprocess.run([cc, std, "-Wall", "-Wextra", "-pedantic", "-Werror", "-fsyntax-only", "-I", str(ROOT / "include"), str(src)],
                           capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
    text = (ROOT / "include" / "epilogos_b200.h").read_text()
    assert "torch" not in re.sub(r"/\*.*?\*/", "", text, flags=re.S) and "#include <cuda" not in text
