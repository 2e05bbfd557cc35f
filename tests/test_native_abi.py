"""The C-ABI library builds for sm_100a, loads, and exports every symbol that
include/gfx.h declares.  No compute calls here (no GPU on the CPU runner);
argument checking that happens before any CUDA call is exercised."""
import ctypes
import re
import shutil
import subprocess
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parents[1]
LIB = ROOT / "ginfinity_b200" / "libgfx.so"


@pytest.fixture(scope="module")
def nat():
    from ginfinity_b200 import build_native
    if not LIB.is_file() and shutil.which(build_native.NVCC) is None:
        pytest.skip("libgfx.so is not built and nvcc is not installed here")
    if shutil.which(build_native.NVCC) is not None:
        build_native.build()
    from ginfinity_b200 import _native
    return _native


def declared_symbols():
    text = (ROOT / "include" / "gfx.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(gfx_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_are_exported(nat):
    names = declared_symbols()
    assert len(names) >= 18
    for name in names:
        assert hasattr(nat.lib, name), f"{name} declared in gfx.h but not exported"
    assert sorted(nat.EXPORTED_SYMBOLS) == names     # binding covers the whole header
    assert nat.lib.gfx_abi_version() == 1


def test_signatures_use_plain_c_types_only():
    text = (ROOT / "include" / "gfx.h").read_text()
    assert "torch" not in text.lower().replace("no torch", "") and "std::" not in text
    assert 'extern "C"' in text


@pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump is not installed here")
def test_library_is_sm_100a_and_uses_the_blackwell_units(nat):
    lib = LIB
    elf = subprocess.run(["cuobjdump", "-lelf", str(lib)], capture_output=True, text=True).stdout
    assert "sm_100a" in elf
    sass = subprocess.run(["cuobjdump", "-sass", str(lib)], capture_output=True, text=True).stdout
    assert "UTCHMMA" in sass          # tcgen05.mma kind::f16
    assert "LDTM" in sass             # tcgen05.ld
    assert "UBLKCP" in sass           # bulk async copy (TMA engine)
    assert "HMMA." not in sass.replace("UTCHMMA", "")   # no legacy mma.sync path
    assert "UTMALDG.2D" in sass and "UTMASTG.2D" in sass   # 2-D tiled TMA loads and stores
    assert "UTCHMMA.2CTA" in sass      # tcgen05.mma.cta_group::2 (fused layer on CTA pairs)
    assert "UTCBAR.2CTA.MULTICAST" in sass   # tcgen05.commit multicast to both CTAs of a pair
    assert "STTM" in sass              # tcgen05.st: the hidden activation goes back into TMEM


def _kernels_sass(sass: str, needle: str) -> list:
    """SASS text of every kernel whose (mangled) name contains `needle`."""
    parts = sass.split("Function : ")
    return [p for p in parts if needle in p.split("\n", 1)[0]]


def _kernel_sass(sass: str, needle: str) -> str:
    """SASS text of the first kernel whose (mangled) name contains `needle`."""
    body = _kernels_sass(sass, needle)
    assert body, needle
    return body[0]


@pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump is not installed here")
def test_each_layer_kernel_is_one_build_with_uniform_issuers(nat):
    """The layer kernels follow their executed-instruction count (DESIGN.md 9.1): each is built
    once, with no timeline stamps, and the banded kernel's MMA / TMA issuers must be
    warp-converged with one elected lane -- issued from inside `if (lane == 0)` every
    tcgen05.mma / TMA instruction comes wrapped in an ELECT / R2UR.BROADCAST / BRA.U.ANY loop."""
    sass = subprocess.run(["cuobjdump", "-sass", str(LIB)], capture_output=True, text=True).stdout
    banded = _kernels_sass(sass, "fused_banded8_kernel")
    pair = _kernels_sass(sass, "fused_pair_kernel")
    assert len(banded) == 1 and len(pair) == 1
    for body in banded + pair:
        assert "SR_CLOCKLO" not in body and "SR_GLOBALTIMER" not in body
    assert banded[0].count("UTCHMMA.2CTA") == 24           # 8 (GEMM 1, N = 256) + 16 (GEMM 2)
    assert pair[0].count("UTCHMMA.2CTA") == 24             # the same GEMMs
    assert "R2UR.BROADCAST" not in banded[0]
    # the same for the top-k scan's MMA issuer
    scan = _kernel_sass(sass, "topk_scan")
    assert scan.count("R2UR.BROADCAST") <= 2 * scan.count("UTMALDG")   # none left around the MMAs


def test_library_reads_no_environment():
    """Which kernel runs, and what it computes, depends on the arguments alone: no source file of
    the library reads an environment variable."""
    readers = [path.name for path in sorted((ROOT / "ginfinity_b200" / "csrc").glob("*.cu*"))
               if "getenv" in path.read_text()]
    assert readers == []


def test_argument_errors_surface_through_gfx_last_error(nat):
    rc = nat.lib.gfx_pack_microbatches(None, None, 0, 10, 10, None, None, None, None)
    assert rc != 0 and b"empty" in nat.lib.gfx_last_error()
    rc = nat.lib.gfx_pack_microbatches(None, None, 5, 0, 10, None, None, None, None)
    assert rc != 0 and b"positive" in nat.lib.gfx_last_error()
    with pytest.raises(nat.NativeError, match="null model"):
        nat.check(nat.lib.gfx_encode(None, None, None, None, None, None, 1, None, 0, 0, 0, 0,
                                     None, 0, None))
    assert nat.lib.gfx_csr_workspace_bytes(1000, 5000) >= 4 * 1001 + 4 * 5000
    assert nat.lib.gfx_encode_workspace_bytes(1000, 0) >= 3 * 1000 * 128 * 2


def test_missing_library_fails_loudly(tmp_path, monkeypatch):
    """No silent fallback: without libgfx.so the binding cannot be imported."""
    import importlib.util
    src = (ROOT / "ginfinity_b200" / "_native.py").read_text()
    fake = tmp_path / "_native_copy.py"
    fake.write_text(src)
    spec = importlib.util.spec_from_file_location("_native_copy", fake)
    module = importlib.util.module_from_spec(spec)
    with pytest.raises(ImportError, match="has not been built"):
        spec.loader.exec_module(module)
