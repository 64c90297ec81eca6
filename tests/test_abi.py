"""The C-ABI library loads and exports every symbol include/zstd_b200.h declares (no compute call:
this runs on the CPU-only box), and the non-compute helpers behave like the reference's."""
import ctypes
import os
import re

import pytest

import zref
import zstd_b200

HEADER = os.path.join(zref.ROOT, "include", "zstd_b200.h")


def declared_symbols():
    text = open(HEADER).read()
    return sorted(set(re.findall(r"ZSTDB200_API\s+[\w\s\*]+?\b(ZSTD\w+)\s*\(", text)))


def test_header_declares_the_reference_entry_points():
    syms = declared_symbols()
    for s in ("ZSTD_compress", "ZSTD_compressCCtx", "ZSTD_compress_usingDict", "ZSTD_createCCtx", "ZSTD_freeCCtx",
              "ZSTD_compressBound", "ZSTD_isError", "ZSTD_getErrorName", "ZSTD_getErrorCode",
              "ZSTD_minCLevel", "ZSTD_maxCLevel", "ZSTD_defaultCLevel", "ZSTD_versionNumber"):
        assert s in syms


def test_library_exports_every_declared_symbol():
    L = ctypes.CDLL(zstd_b200.LIB_PATH, mode=ctypes.RTLD_LOCAL)
    for s in declared_symbols():
        assert hasattr(L, s), f"{s} declared in include/zstd_b200.h but not exported"


def test_helpers_match_reference_semantics():
    L = zstd_b200.lib()
    assert L.ZSTD_versionNumber() == 10506
    assert L.ZSTD_minCLevel() == -(1 << 17) and L.ZSTD_maxCLevel() == 22 and L.ZSTD_defaultCLevel() == 3
    assert L.ZSTD_freeCCtx(None) == 0                                   # lib/zstd.h:264 accepts NULL
    for n in [0, 1, 100, 128 << 10, (128 << 10) + 1, 1 << 30]:
        assert L.ZSTD_compressBound(n) == zref.oracle().zbo_compressBound(n)
    assert L.ZSTD_isError(L.ZSTD_compressBound(0xFF00FF00FF00FF00))      # srcSize_wrong
    assert L.ZSTD_getErrorCode(L.ZSTD_compressBound(0xFF00FF00FF00FF00)) == 72
    assert not L.ZSTD_isError(12345)
    for code in (0, 1, 10, 30, 32, 40, 42, 44, 46, 60, 62, 64, 66, 70, 72, 74, 119):
        v = (1 << 64) - code if code else 0
        assert L.ZSTD_getErrorName(v).decode() == zref.ref_error_name(v), code
        assert bool(L.ZSTD_isError(v)) == bool(zref.ref_call("ZSTD_isError", v))


def test_context_lifecycle_without_gpu():
    L = zstd_b200.lib()
    c = L.ZSTD_createCCtx()
    assert c
    assert L.ZSTD_freeCCtx(c) == 0


@pytest.mark.skipif(zstd_b200.device_available(), reason="CUDA device present")
def test_compress_fails_loudly_without_cuda():
    """No CPU fallback: without a device the call must return an error, never data."""
    with pytest.raises(zstd_b200.ZstdError):
        zstd_b200.ZSTD_compress(b"hello world" * 100, 1)


def test_header_is_valid_c99_and_links(tmp_path):
    """A C caller (what INTEGRATION.md shows) compiles against include/zstd_b200.h with a C99 compiler and links against
    the shared library without a GPU present (no call is made)."""
    import os, shutil, subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = tmp_path / "caller.c"
    src.write_text('#include "zstd_b200.h"\n'
                   '#include <stdio.h>\n'
                   'int main(int argc, char** argv) {\n'
                   '    if (argc > 1000) {  /* never true: only the link matters */\n'
                   '        ZSTD_CCtx* c = ZSTD_createCCtx(); ZSTD_CDict* d = ZSTD_createCDict(argv[0], 8, 1); char dst[64];\n'
                   '        ZSTD_CCtx_setParameter(c, ZSTD_c_checksumFlag, 1);\n'
                   '        printf("%zu %zu %zu\\n", ZSTD_compress2(c, dst, sizeof dst, argv[0], 4), ZSTD_compress_usingCDict(c, dst, sizeof dst, argv[0], 4, d),\n'
                   '               ZSTD_compress(dst, sizeof dst, argv[0], 4, 1));\n'
                   '        ZSTD_freeCDict(d); ZSTD_freeCCtx(c);\n'
                   '    }\n'
                   '    printf("%u %s\\n", ZSTD_versionNumber(), ZSTD_getErrorName((size_t)-70));\n'
                   '    return 0;\n}\n')
    gcc = shutil.which("gcc")
    if not gcc:
        pytest.skip("no gcc")
    exe = tmp_path / "caller"
    libdir = os.path.join(root, "zstd_b200")
    cmd = [gcc, "-std=c99", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I", os.path.join(root, "include"), str(src), "-o", str(exe),
           "-L", libdir, "-lzstd_b200", "-Wl,-rpath," + libdir, "-L/usr/local/cuda/lib64", "-Wl,-rpath,/usr/local/cuda/lib64"]
    subprocess.check_call(cmd)
    out = subprocess.check_output([str(exe)], text=True)
    assert out.split()[0] == "10506" and "too small" in out


def test_soname_build_target(tmp_path):
    """`make -C zstd_b200/csrc soname` produces the same code under the reference's shared-library name (lib/Makefile:85,145)"""
    import shutil, subprocess
    if not shutil.which("nvcc") or not shutil.which("readelf"):
        pytest.skip("no nvcc / readelf")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    subprocess.check_call(["make", "-s", "-C", os.path.join(root, "zstd_b200", "csrc"), "soname"])
    out = subprocess.check_output(["readelf", "-d", os.path.join(root, "zstd_b200", "libzstd.so.1")], text=True)
    assert "libzstd.so.1" in out and "SONAME" in out
