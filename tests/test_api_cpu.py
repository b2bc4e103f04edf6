"""CPU tests of the boundary: the C-ABI library loads and exports everything include/*.h declares,
liblzma struct layouts match the reference headers, option validation returns liblzma's codes
(no compute calls -- there is no GPU here, and no CPU fallback to call)."""
import ctypes as C
import hashlib
import json
import os
import re
import subprocess

import pytest

import xzlibs as X

ROOT = X.ROOT


def _declared(header):
    txt = open(os.path.join(ROOT, "include", header)).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b((?:xzb|lzma)_[a-z0-9_]+)\s*\(", txt)) - {"lzma_internal_s"})


def test_library_exports_every_declared_symbol():
    import xz_b200
    lib = xz_b200.lib()
    names = _declared("xzb200.h") + _declared("xzb200_lzma.h")
    assert len(names) > 25
    for n in names:
        assert hasattr(lib, n), n


def test_no_gpu_fails_loudly():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import xz_b200
    with pytest.raises(xz_b200.XzError):
        xz_b200.Context(0)


LAYOUT_PROG = r'''
#include <stdio.h>
#include <stddef.h>
#include HEADER
#define P(T, f) printf(#T "." #f " %zu %zu\n", offsetof(T, f), sizeof(((T *)0)->f))
int main(void) {
	printf("sizeof %zu %zu %zu %zu %zu\n", sizeof(lzma_stream), sizeof(lzma_mt), sizeof(lzma_options_lzma), sizeof(lzma_filter), sizeof(lzma_allocator));
	P(lzma_stream, next_in); P(lzma_stream, avail_in); P(lzma_stream, total_in); P(lzma_stream, next_out); P(lzma_stream, avail_out);
	P(lzma_stream, total_out); P(lzma_stream, allocator); P(lzma_stream, internal); P(lzma_stream, seek_pos); P(lzma_stream, reserved_enum2);
	P(lzma_mt, flags); P(lzma_mt, threads); P(lzma_mt, block_size); P(lzma_mt, timeout); P(lzma_mt, preset); P(lzma_mt, filters); P(lzma_mt, check);
	P(lzma_mt, memlimit_threading); P(lzma_mt, memlimit_stop); P(lzma_mt, reserved_ptr4);
	P(lzma_options_lzma, dict_size); P(lzma_options_lzma, preset_dict); P(lzma_options_lzma, preset_dict_size); P(lzma_options_lzma, lc);
	P(lzma_options_lzma, lp); P(lzma_options_lzma, pb); P(lzma_options_lzma, mode); P(lzma_options_lzma, nice_len); P(lzma_options_lzma, mf);
	P(lzma_options_lzma, depth); P(lzma_options_lzma, ext_flags); P(lzma_options_lzma, reserved_ptr2);
	P(lzma_filter, id); P(lzma_filter, options);
	printf("sizeof lzma_block %zu\n", sizeof(lzma_block));
	P(lzma_block, version); P(lzma_block, header_size); P(lzma_block, check); P(lzma_block, compressed_size); P(lzma_block, uncompressed_size);
	P(lzma_block, filters); P(lzma_block, raw_check); P(lzma_block, reserved_ptr1); P(lzma_block, reserved_int3); P(lzma_block, reserved_enum1);
	P(lzma_block, ignore_check); P(lzma_block, reserved_bool8);
	printf("enums %d %d %d %d %d %d %d %d\n", LZMA_FINISH, LZMA_FULL_BARRIER, LZMA_FULL_FLUSH, LZMA_BUF_ERROR, LZMA_PROG_ERROR, LZMA_CHECK_CRC64, LZMA_MF_BT4, LZMA_MODE_NORMAL);
	return 0;
}
'''


def test_struct_layouts_match_reference_headers(tmp_path):
    """The probe compiled against include/xzb200_lzma.h prints what it printed against the reference's <lzma.h>
    (recorded in tests/golden/ref_checks_golden.json)."""
    src = tmp_path / "l.c"
    src.write_text(LAYOUT_PROG.replace("HEADER", '"xzb200_lzma.h"'))
    exe = tmp_path / "l"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    assert subprocess.check_output([str(exe)], text=True) == X.ref_golden()["lzma_h_layout"]


class LzmaStream(C.Structure):
    _fields_ = [("next_in", C.c_void_p), ("avail_in", C.c_size_t), ("total_in", C.c_uint64), ("next_out", C.c_void_p),
                ("avail_out", C.c_size_t), ("total_out", C.c_uint64), ("allocator", C.c_void_p), ("internal", C.c_void_p),
                ("reserved_ptr1", C.c_void_p), ("reserved_ptr2", C.c_void_p), ("reserved_ptr3", C.c_void_p), ("reserved_ptr4", C.c_void_p),
                ("seek_pos", C.c_uint64), ("reserved_int2", C.c_uint64), ("reserved_int3", C.c_size_t), ("reserved_int4", C.c_size_t),
                ("reserved_enum1", C.c_int), ("reserved_enum2", C.c_int)]


class LzmaMt(C.Structure):
    _fields_ = [("flags", C.c_uint32), ("threads", C.c_uint32), ("block_size", C.c_uint64), ("timeout", C.c_uint32), ("preset", C.c_uint32),
                ("filters", C.c_void_p), ("check", C.c_int), ("reserved_enum1", C.c_int), ("reserved_enum2", C.c_int), ("reserved_enum3", C.c_int),
                ("reserved_int1", C.c_uint32), ("reserved_int2", C.c_uint32), ("reserved_int3", C.c_uint32), ("reserved_int4", C.c_uint32),
                ("memlimit_threading", C.c_uint64), ("memlimit_stop", C.c_uint64), ("reserved_int7", C.c_uint64), ("reserved_int8", C.c_uint64),
                ("reserved_ptr1", C.c_void_p), ("reserved_ptr2", C.c_void_p), ("reserved_ptr3", C.c_void_p), ("reserved_ptr4", C.c_void_p)]


class LzmaFilter(C.Structure):
    _fields_ = [("id", C.c_uint64), ("options", C.c_void_p)]


class LzmaOptionsLzma(C.Structure):
    _fields_ = [("dict_size", C.c_uint32), ("preset_dict", C.c_void_p), ("preset_dict_size", C.c_uint32), ("lc", C.c_uint32), ("lp", C.c_uint32),
                ("pb", C.c_uint32), ("mode", C.c_int), ("nice_len", C.c_uint32), ("mf", C.c_int), ("depth", C.c_uint32), ("ext_flags", C.c_uint32),
                ("ext_size_low", C.c_uint32), ("ext_size_high", C.c_uint32), ("reserved_int4", C.c_uint32), ("reserved_int5", C.c_uint32),
                ("reserved_int6", C.c_uint32), ("reserved_int7", C.c_uint32), ("reserved_int8", C.c_uint32), ("reserved_enum1", C.c_int),
                ("reserved_enum2", C.c_int), ("reserved_enum3", C.c_int), ("reserved_enum4", C.c_int), ("reserved_ptr1", C.c_void_p),
                ("reserved_ptr2", C.c_void_p)]


class LzmaBlock(C.Structure):
    _fields_ = [("version", C.c_uint32), ("header_size", C.c_uint32), ("check", C.c_int), ("compressed_size", C.c_uint64),
                ("uncompressed_size", C.c_uint64), ("filters", C.c_void_p), ("raw_check", C.c_uint8 * 64), ("reserved_ptr", C.c_void_p * 3),
                ("reserved_int12", C.c_uint32 * 2), ("reserved_int38", C.c_uint64 * 6), ("reserved_enum", C.c_int * 4), ("bools", C.c_uint8 * 8)]


def _mt(**kw):
    m = LzmaMt()
    m.threads, m.preset, m.check, m.block_size = 1, 6, 4, 1 << 20
    for k, v in kw.items():
        setattr(m, k, v)
    return m


BAD_OPTIONS = [({"flags": 1}, 8), ({"threads": 0}, 8), ({"threads": 20000}, 8), ({"preset": 10}, 8), ({"preset": 6 | 0x40000000}, 8),
               ({"check": 10}, 0), ({"check": 2}, 3), ({"check": 16}, 11), ({"block_size": (1 << 64) - 1}, 8)]


@pytest.mark.parametrize("kw,want", BAD_OPTIONS)
def test_encoder_mt_option_validation(kw, want):
    """lzma_stream_encoder_mt rejects bad lzma_mt fields with the reference's codes
    (stream_encoder_mt.c:955-1000, 1052-1060) before any device work."""
    import xz_b200
    lib = xz_b200.lib()
    s = LzmaStream()
    m = _mt(**kw)
    got = lib.lzma_stream_encoder_mt(C.byref(s), C.byref(m))
    assert X.ref_golden()["mt_options"][json.dumps(kw, sort_keys=True)] == want
    import torch
    if want == 0 and not torch.cuda.is_available():
        assert got not in (0, 1)  # valid options, but no GPU: fails loudly when the context is created
    else:
        assert got == want
    lib.lzma_end(C.byref(s))
    assert not s.internal


def test_lzma_code_argument_checks_without_coder():
    import xz_b200
    lib = xz_b200.lib()
    s = LzmaStream()
    assert lib.lzma_code(C.byref(s), 0) == 11  # internal == NULL -> LZMA_PROG_ERROR (common.c:206-213)
    lib.lzma_end(C.byref(s))  # no-op on a fresh stream


def test_preset_table_matches_oracle():
    import xz_b200
    for p in list(range(10)) + [i | 0x80000000 for i in range(10)]:
        a, b = xz_b200.lzma_lzma_preset(p), X.preset_options(p)
        assert [getattr(a, f) for f, _ in a._fields_] == [getattr(b, f) for f, _ in b._fields_]
    assert xz_b200.lib().xzb_block_bound(1 << 24) == X.oracle().xzo_block_bound(1 << 24) == 16778080


def test_framing_helpers_match_oracle():
    """Stream Header / Index / Footer built by the product's host code == oracle's."""
    import xz_b200
    recs = [(16778072, 1 << 24), (100, 5), (70000, 1 << 20), (3000005, 1 << 24)]
    idx = xz_b200.index_encode(recs)
    U = (C.c_uint64 * len(recs))(*[r[0] for r in recs])
    V = (C.c_uint64 * len(recs))(*[r[1] for r in recs])
    o = X.oracle()
    o.xzo_index_encode.restype = C.c_size_t
    n = o.xzo_index_encode(U, V, C.c_size_t(len(recs)), None)
    buf = (C.c_uint8 * n)()
    o.xzo_index_encode(U, V, C.c_size_t(len(recs)), buf)
    assert idx == bytes(buf)
    hdr = (C.c_uint8 * 12)(); o.xzo_stream_header(hdr, C.c_uint32(4))
    ftr = (C.c_uint8 * 12)(); o.xzo_stream_footer(ftr, C.c_uint32(4), C.c_uint64(len(idx)))
    assert xz_b200.stream_header(4) == bytes(hdr) and xz_b200.stream_footer(4, len(idx)) == bytes(ftr)


def test_buffer_bounds_match_reference_golden():
    """lzma_stream_buffer_bound / lzma_block_buffer_bound incl. the overflow rules
    (stream_buffer_encoder.c:17-40, block_buffer_encoder.c:31-84)."""
    import json
    import xz_b200
    lib = xz_b200.lib()
    lib.lzma_stream_buffer_bound.restype = C.c_size_t
    lib.lzma_stream_buffer_bound.argtypes = [C.c_size_t]
    lib.lzma_block_buffer_bound.restype = C.c_size_t
    lib.lzma_block_buffer_bound.argtypes = [C.c_size_t]
    g = json.load(open(os.path.join(ROOT, "tests", "golden", "buffer_golden.json")))["stream_buffer_bound"]
    for k, v in g.items():
        assert lib.lzma_stream_buffer_bound(int(k)) == v, k
        assert lib.lzma_block_buffer_bound(int(k)) == (v - 48 if v else 0), k


def test_buffer_api_argument_checks_need_no_gpu():
    """The argument checks of stream_buffer_encoder.c:49-68 / stream_buffer_decoder.c:20-29 come before
    any device work; with valid arguments and no GPU the call fails loudly (no CPU fallback)."""
    import torch
    import xz_b200
    lib = xz_b200.lib()
    out = (C.c_uint8 * 4096)()
    pos = C.c_size_t(0)
    enc = lambda preset, check, data, n, op, cap: lib.lzma_easy_buffer_encode(C.c_uint32(preset), C.c_int(check), None, data, C.c_size_t(n),
                                                                               out, op, C.c_size_t(cap))
    assert enc(6, 4, b"abc", 3, None, 4096) == 11          # out_pos == NULL
    assert enc(6, 4, None, 3, C.byref(pos), 4096) == 11    # in == NULL with in_size != 0
    assert enc(6, 16, b"abc", 3, C.byref(pos), 4096) == 11  # check > LZMA_CHECK_ID_MAX
    assert enc(6, 2, b"abc", 3, C.byref(pos), 4096) == 3   # LZMA_UNSUPPORTED_CHECK
    assert enc(10, 4, b"abc", 3, C.byref(pos), 4096) == 8  # bad preset
    assert enc(6, 4, b"abc", 3, C.byref(pos), 24) == 10    # no room for Stream Header + Footer
    pos.value = 5000
    assert enc(6, 4, b"abc", 3, C.byref(pos), 4096) == 11  # *out_pos > out_size
    ip, op = C.c_size_t(0), C.c_size_t(0)
    ml = C.c_uint64((1 << 64) - 1)
    dec = lambda flags, ipp, n: lib.lzma_stream_buffer_decode(C.byref(ml), C.c_uint32(flags), None, b"\xfd7zXZ\0" + bytes(26), ipp, C.c_size_t(n),
                                                               out, C.byref(op), C.c_size_t(4096))
    assert dec(0x04, C.byref(ip), 32) == 11  # LZMA_TELL_ANY_CHECK is not allowed here
    assert dec(0x40, C.byref(ip), 32) == 8   # unknown flag
    assert dec(0, None, 32) == 11
    ip.value = 33
    assert dec(0, C.byref(ip), 32) == 11
    if not torch.cuda.is_available():
        pos.value = 0
        assert enc(6, 4, b"abc", 3, C.byref(pos), 4096) not in (0, 1) and pos.value == 0
        ip.value = 0
        assert dec(0, C.byref(ip), 32) not in (0, 1)


def test_block_buffer_encode_empty_input_and_argument_checks():
    """lzma_block_buffer_encode: the argument checks of block_buffer_encoder.c:219-252 and the one case that needs no
    device work (zero bytes of input: header + LZMA2 end marker + check of nothing) against the reference's bytes."""
    import json
    import xz_b200
    lib = xz_b200.lib()
    gold = json.load(open(os.path.join(ROOT, "tests", "golden", "buffer_golden.json")))["block_buffer_encode"]
    o = LzmaOptionsLzma()
    assert lib.lzma_lzma_preset(C.byref(o), C.c_uint32(6)) == 0
    f = (LzmaFilter * 2)()
    f[0].id, f[0].options = 0x21, C.cast(C.pointer(o), C.c_void_p)
    f[1].id = (1 << 64) - 1
    out = (C.c_uint8 * 256)()
    for g in [c for c in gold if c["size"] == 0]:
        b = LzmaBlock(); b.check, b.filters = g["check"], C.cast(f, C.c_void_p)
        pos = C.c_size_t(0)
        assert lib.lzma_block_buffer_encode(C.byref(b), None, None, C.c_size_t(0), out, C.byref(pos), C.c_size_t(256)) == 0
        blk = bytes(out[: pos.value])
        assert len(blk) == g["block_size"] and hashlib.sha256(blk).hexdigest() == g["block_sha256"]
        assert (b.header_size, b.compressed_size, b.uncompressed_size) == (g["header_size"], g["compressed_size"], 0)
        assert bytes(b.raw_check).hex()[: 2 * {0: 0, 1: 4, 4: 8, 10: 32}[g["check"]]] == g["raw_check"][: 2 * {0: 0, 1: 4, 4: 8, 10: 32}[g["check"]]]
    b = LzmaBlock(); b.check, b.filters = 4, C.cast(f, C.c_void_p)
    pos = C.c_size_t(0)
    enc = lambda blk, n, op, cap: lib.lzma_block_buffer_encode(blk, None, b"abc", C.c_size_t(n), out, op, C.c_size_t(cap))
    assert enc(None, 3, C.byref(pos), 256) == 11
    assert enc(C.byref(b), 3, None, 256) == 11
    assert enc(C.byref(b), 3, C.byref(pos), 8) == 10   # no room beyond the Check field
    b.version = 2
    assert enc(C.byref(b), 3, C.byref(pos), 256) == 8
    b.version, b.check = 0, 16
    assert enc(C.byref(b), 3, C.byref(pos), 256) == 11
    b.check = 3
    assert enc(C.byref(b), 3, C.byref(pos), 256) == 3
    b.check, b.filters = 4, None
    assert enc(C.byref(b), 3, C.byref(pos), 256) == 11
    f[0].id = 0x03  # Delta: not a chain the GPU path takes
    b.filters = C.cast(f, C.c_void_p)
    assert enc(C.byref(b), 3, C.byref(pos), 256) == 8


class LzmaFilter(C.Structure):
    _fields_ = [("id", C.c_uint64), ("options", C.c_void_p)]


class LzmaOptionsDelta(C.Structure):
    _fields_ = [("type", C.c_int), ("dist", C.c_uint32), ("reserved_int", C.c_uint32 * 4), ("reserved_ptr", C.c_void_p * 2)]


class LzmaOptionsBcj(C.Structure):
    _fields_ = [("start_offset", C.c_uint32)]


def _chain(spec, keep):
    """spec: list of (id, arg) with id 0x21 = LZMA2 (preset 6); returns a lzma_filter array (keep holds the option structs)."""
    import xz_b200
    arr = (LzmaFilter * (len(spec) + 1))()
    for i, (fid, arg) in enumerate(spec):
        arr[i].id = fid
        if fid == 0x21:
            o = LzmaOptionsLzma()
            p = xz_b200.lzma_lzma_preset(6)
            o.dict_size, o.lc, o.lp, o.pb, o.mode, o.nice_len, o.mf, o.depth = p.dict_size, p.lc, p.lp, p.pb, p.mode, p.nice_len, p.mf, p.depth
        elif fid == 0x03:
            o = LzmaOptionsDelta(); o.type = 0; o.dist = arg
        else:
            o = LzmaOptionsBcj(); o.start_offset = arg
        keep.append(o)
        arr[i].options = C.cast(C.pointer(o), C.c_void_p)
    arr[len(spec)].id = (1 << 64) - 1
    return arr


BAD_CHAINS = [[(0x04, 0)], [(0x21, 0), (0x04, 0)], [(0x03, 0), (0x21, 0)], [(0x03, 257), (0x21, 0)],
              [(0x0C, 0), (0x21, 0)], [(0x04, 0), (0x03, 1), (0x07, 0), (0x0A, 0), (0x21, 0)], [(0x21, 0), (0x21, 0)]]
# (a misaligned BCJ start offset passes lzma_stream_encoder_mt in the reference and fails in lzma_code: tests/test_gpu_lzma_api.py)
GOOD_CHAINS = [[(0x21, 0)], [(0x04, 0), (0x21, 0)], [(0x03, 256), (0x0B, 0x1002), (0x21, 0)], [(0x06, 32), (0x09, 4), (0x05, 8), (0x21, 0)],
               [(0x07, 2), (0x21, 0)], [(0x06, 8), (0x21, 0)], [(0x0B, 1), (0x21, 0)]]


def chain_id(spec):
    return "+".join(f"{i:x}.{a:x}" for i, a in spec)


@pytest.mark.parametrize("spec", BAD_CHAINS + GOOD_CHAINS, ids=chain_id)
def test_filter_chain_validation_matches_reference(spec):
    """lzma_stream_encoder_mt with lzma_mt.filters: chains the table common/filter_encoder.c:59-182 refuses (LZMA2 not last,
    too many filters, unknown IDs, Delta distance, BCJ start-offset alignment) get LZMA_OPTIONS_ERROR before any device
    work, like the reference; valid chains pass validation (and then need the GPU).  lzma_mt_block_size agrees too."""
    import xz_b200
    lib = xz_b200.lib()
    lib.lzma_mt_block_size.restype = C.c_uint64
    keep = []
    arr = _chain(spec, keep)
    m = _mt(filters=C.cast(arr, C.c_void_p))
    s = LzmaStream()
    got = lib.lzma_stream_encoder_mt(C.byref(s), C.byref(m))
    lib.lzma_end(C.byref(s))
    bad = spec in BAD_CHAINS
    ref = X.ref_golden()["filter_chains"][chain_id(spec)]
    assert (ref["ret"] != 0) == bad, (spec, ref["ret"])
    if not bad:
        assert lib.lzma_mt_block_size(arr) == ref["mt_block_size"]
    import torch
    if bad:
        assert got == 8, (spec, got)
    elif not torch.cuda.is_available():
        assert got not in (0, 1, 8), (spec, got)   # valid chain, no GPU: the context creation fails loudly
    else:
        assert got == 0
