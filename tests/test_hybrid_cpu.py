"""The drop-in boundary under the UNMODIFIED reference `xz` (src/xz, built by oracle/Makefile.ref): CPU-side checks.

oracle/_ref/xz      = reference xz + reference liblzma                       (the binary to compare with)
oracle/_ref/xz_gpu  = the same objects with libxzb200.so ahead of liblzma    (the hybrid of INTEGRATION.md)

No GPU work here: layout of lzma_stream.internal against the reference header, symbol resolution of the hybrid,
the reference's own coders driven through this library's generic lzma_code, and the loud failure without CUDA."""
import os
import re
import subprocess

import pytest

import xzlibs as X

ROOT = X.ROOT
XZ = os.path.join(ROOT, "oracle", "_ref", "xz")
XZ_GPU = os.path.join(ROOT, "oracle", "_ref", "xz_gpu")
needs_bins = pytest.mark.skipif(not (os.path.exists(XZ) and os.path.exists(XZ_GPU)), reason="oracle/_ref/xz[_gpu] not built")


def test_internal_layout_matches_reference_header(tmp_path):
    """xzb_lzma_api.cpp restates lzma_next_coder_s / lzma_internal_s (common/common.h:222-324); a probe compiled against
    that restatement must report the offsets a probe compiled against the reference's own common.h reported (below:
    the 11 of lzma_next_coder, the 6 of lzma_internal, LZMA_ACTION_MAX; the reference's probe also gave LZMA_TIMED_OUT = 101)."""
    shim = open(os.path.join(ROOT, "xz_b200", "csrc", "xzb_lzma_api.cpp")).read()
    structs = re.search(r"^struct xzb_next_coder \{.*?^\};\nstruct lzma_internal_s \{.*?^\};\n", shim, re.S | re.M).group(0)
    src = tmp_path / "probe.cpp"
    src.write_text('#include <cstdio>\n#include <cstddef>\n#include "xzb200_lzma.h"\n' + structs + r'''
int main(void) {
	printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu ", offsetof(xzb_next_coder, coder), offsetof(xzb_next_coder, id),
		offsetof(xzb_next_coder, init), offsetof(xzb_next_coder, code), offsetof(xzb_next_coder, end),
		offsetof(xzb_next_coder, get_progress), offsetof(xzb_next_coder, get_check), offsetof(xzb_next_coder, memconfig),
		offsetof(xzb_next_coder, update), offsetof(xzb_next_coder, set_out_limit), sizeof(xzb_next_coder));
	printf("%zu %zu %zu %zu %zu %zu %zu\n", offsetof(lzma_internal_s, next), offsetof(lzma_internal_s, sequence),
		offsetof(lzma_internal_s, avail_in), offsetof(lzma_internal_s, supported_actions), offsetof(lzma_internal_s, allow_buf_error),
		sizeof(lzma_internal_s), sizeof(((lzma_internal_s *)0)->supported_actions) - 1);
	return 0;
}''')
    exe = tmp_path / "probe"
    subprocess.run(["g++", "-std=c++17", f"-I{ROOT}/include", str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], stdout=subprocess.PIPE, text=True, check=True).stdout.split()]
    assert got == [0, 8, 16, 24, 32, 40, 48, 56, 64, 72, 80, 0, 80, 88, 96, 101, 104, 4]
    assert re.search(r"^\tcase 101:  // LZMA_TIMED_OUT", shim, re.M)   # LZMA_TIMED_OUT = 101


def test_hybrid_resolves_every_symbol_xz_imports():
    """Every lzma_* symbol the unmodified xz imports is defined by libxzb200.so or by the reference liblzma behind it
    (both symbol lists recorded from the reference build in tests/golden/ref_checks_golden.json)."""
    def syms(path, flag):
        out = subprocess.run(["nm", "-D", flag, path], stdout=subprocess.PIPE, text=True, check=True).stdout
        return {ln.split()[-1] for ln in out.splitlines() if re.search(r"\blzma_", ln)}
    imports = set(X.ref_golden()["xz_imports"])
    ours = syms(os.path.join(ROOT, "xz_b200", "libxzb200.so"), "--defined-only")
    theirs = set(X.ref_golden()["ref_liblzma_exports"])
    assert len(imports) >= 37
    assert imports <= (ours | theirs), sorted(imports - ours - theirs)
    # the stream coders of the hot path and the generic drivers come from this library
    for name in ("lzma_stream_encoder_mt", "lzma_stream_decoder_mt", "lzma_code", "lzma_end", "lzma_memusage", "lzma_get_progress",
                 "lzma_filters_update", "lzma_stream_encoder_mt_memusage", "lzma_mt_block_size"):
        assert name in ours and name in imports | ours
    if os.path.exists(XZ_GPU):
        assert imports == syms(XZ_GPU, "--undefined-only")
        out = subprocess.run(["ldd", XZ_GPU], stdout=subprocess.PIPE, text=True).stdout
        assert out.index("libxzb200.so") < out.index("liblzma_ref.so")   # lookup order = link order


@needs_bins
def test_reference_coders_run_through_this_librarys_lzma_code(tmp_path):
    """In the hybrid, lzma_code/lzma_end bind to libxzb200.so.  They are generic over the reference's coder vtable, so the
    reference's single-threaded .xz encoder, its .lzma coders and its file-info decoder (xz -l) behave exactly as under
    the reference's own lzma_code -- byte-identical output, no GPU involved."""
    buf = X.gendata("T", 600000)
    f = tmp_path / "in.bin"
    f.write_bytes(bytes(buf[:600000]))
    a = subprocess.run([XZ, "-6", "-T1", "-c", str(f)], stdout=subprocess.PIPE, check=True).stdout
    b = subprocess.run([XZ_GPU, "-6", "-T1", "-c", str(f)], stdout=subprocess.PIPE, check=True).stdout
    assert a == b
    a = subprocess.run([XZ, "--format=lzma", "-c", str(f)], stdout=subprocess.PIPE, check=True).stdout
    b = subprocess.run([XZ_GPU, "--format=lzma", "-c", str(f)], stdout=subprocess.PIPE, check=True).stdout
    assert a == b
    back = subprocess.run([XZ_GPU, "--format=lzma", "-dc"], input=b, stdout=subprocess.PIPE, check=True).stdout
    assert back == f.read_bytes()
    g = tmp_path / "x.xz"
    g.write_bytes(subprocess.run([XZ, "-6", "-T1", "-c", str(f)], stdout=subprocess.PIPE, check=True).stdout)
    la = subprocess.run([XZ, "-l", str(g)], stdout=subprocess.PIPE, text=True, check=True).stdout
    lb = subprocess.run([XZ_GPU, "-l", str(g)], stdout=subprocess.PIPE, text=True, check=True).stdout
    assert la == lb


@needs_bins
def test_hybrid_fails_loudly_without_cuda(tmp_path):
    """No CPU fallback: the threaded encoder of the hybrid needs the GPU; without one xz reports an error and exits 1."""
    import xz_b200
    try:
        ctx = xz_b200.Context(0)
        ctx.close()
        pytest.skip("a CUDA device is present")
    except Exception:
        pass
    f = tmp_path / "in.bin"
    f.write_bytes(b"hello " * 1000)
    r = subprocess.run([XZ_GPU, "-6", "-T2", "-c", str(f)], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert r.returncode == 1 and b"no usable CUDA device" in r.stderr and r.stdout == b""
