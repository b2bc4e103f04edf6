"""GPU tests (-m gpu) of the liblzma-named entry points (include/xzb200_lzma.h): the canonical
caller pattern of doc/examples/04_compress_easy_mt.c / src/xz/coder.c:1127-1352 -- lzma_code in a
loop with small in/out buffers -- produces the oracle's bytes; flushing, error latching and
LZMA_BUF_ERROR behave as common/common.c:203-376 prescribes."""
import ctypes as C

import pytest

import xzlibs as X
from test_api_cpu import LzmaMt, LzmaStream

pytestmark = pytest.mark.gpu
RUN, FULL_FLUSH, FINISH, FULL_BARRIER = 0, 2, 3, 4


@pytest.fixture(scope="module")
def lib():
    import xz_b200
    return xz_b200.lib()


def _drive(lib, strm, data, in_chunk, out_chunk, final_action=FINISH, actions=None):
    """Feed `data` in in_chunk pieces, drain through an out_chunk-sized buffer; returns (ret, bytes)."""
    out = bytearray()
    obuf = (C.c_uint8 * out_chunk)()
    ibuf = (C.c_uint8 * max(len(data), 1)).from_buffer_copy(data or b"\0")
    pos = 0
    strm.next_out, strm.avail_out = C.addressof(obuf), out_chunk
    ret = 0
    for _ in range(10_000_000):
        if strm.avail_in == 0 and pos < len(data):
            n = min(in_chunk, len(data) - pos)
            strm.next_in, strm.avail_in = C.addressof(ibuf) + pos, n
            pos += n
        action = final_action if pos == len(data) else RUN
        ret = lib.lzma_code(C.byref(strm), action)
        if strm.avail_out == 0 or ret != 0:
            out += bytes(obuf[: out_chunk - strm.avail_out])
            strm.next_out, strm.avail_out = C.addressof(obuf), out_chunk
        if ret != 0:
            break
    return ret, bytes(out)


@pytest.mark.parametrize("kind,preset,n,bs,inc,outc", [("T", 6, 700001, 1 << 18, 8192, 8192), ("E", 1, 300000, 1 << 16, 1000, 777),
                                                        ("R", 3, 150000, 1 << 16, 150000, 1 << 20), ("T", 1, 0, 1 << 16, 1, 64),
                                                        ("T", 3, 5, 1 << 16, 1, 1)])
def test_stream_encoder_mt_streaming_matches_oracle(lib, kind, preset, n, bs, inc, outc):
    buf = X.gendata(kind, n)
    data = bytes(buf[:n])
    s = LzmaStream()
    m = LzmaMt(); m.threads, m.preset, m.check, m.block_size = 4, preset, 4, bs
    assert lib.lzma_stream_encoder_mt(C.byref(s), C.byref(m)) == 0
    ret, out = _drive(lib, s, data, inc, outc)
    assert ret == 1  # LZMA_STREAM_END
    assert s.total_in == n and s.total_out == len(out)
    assert out == X.oracle_encode(buf, n, preset, bs)
    assert lib.lzma_code(C.byref(s), FINISH) == 1  # ISEQ_END keeps answering LZMA_STREAM_END
    lib.lzma_end(C.byref(s))
    assert not s.internal
    # and back through lzma_stream_decoder with other odd buffer sizes
    d = LzmaStream()
    assert lib.lzma_stream_decoder(C.byref(d), C.c_uint64((1 << 64) - 1), C.c_uint32(0)) == 0
    ret, back = _drive(lib, d, out, 4099, 3001)
    assert ret == 1 and back == data
    lib.lzma_end(C.byref(d))


def test_full_flush_ends_blocks_like_the_reference(lib):
    """LZMA_FULL_FLUSH finishes the pending Block (stream_encoder_mt.c:617-624); three flushed pieces
    of 100000 bytes with a 1 MiB block size give three short Blocks.  Oracle equivalent: encode each
    piece as its own set of Blocks and splice Index/Footer."""
    import xz_b200
    n = 300000
    buf = X.gendata("T", n)
    data = bytes(buf[:n])
    s = LzmaStream()
    m = LzmaMt(); m.threads, m.preset, m.check, m.block_size = 2, 1, 4, 1 << 20
    assert lib.lzma_stream_encoder_mt(C.byref(s), C.byref(m)) == 0
    out = b""
    for i, piece in enumerate((data[:100000], data[100000:200000], data[200000:])):
        ret, o = _drive(lib, s, piece, 50000, 1 << 20, final_action=FULL_FLUSH if i < 2 else FINISH)
        assert ret == 1
        out += o
    lib.lzma_end(C.byref(s))
    r, back = X.oracle_decode(out, n)
    assert r == 0 and back == data
    # three Blocks: compare with oracle-encoded pieces
    blocks, recs = b"", []
    for piece in (data[:100000], data[100000:200000], data[200000:]):
        pb = (C.c_uint8 * len(piece)).from_buffer_copy(piece)
        xz = X.oracle_encode(pb, len(piece), 1, 1 << 20)
        hs = (xz[12] + 1) * 4
        v, sh, p = 0, 0, 14
        while True:
            c = xz[p]; p += 1; v |= (c & 0x7F) << sh; sh += 7
            if not c & 0x80: break
        unp = hs + v + 8
        blocks += xz[12:12 + (unp + 3) // 4 * 4]
        recs.append((unp, len(piece)))
    idx = xz_b200.index_encode(recs)
    assert out == xz_b200.stream_header(4) + blocks + idx + xz_b200.stream_footer(4, len(idx))


def test_lzma_code_sequence_rules(lib):
    s = LzmaStream()
    m = LzmaMt(); m.threads, m.preset, m.check, m.block_size = 1, 1, 4, 1 << 16
    assert lib.lzma_stream_encoder_mt(C.byref(s), C.byref(m)) == 0
    obuf = (C.c_uint8 * 64)()
    ibuf = (C.c_uint8 * 10)(*range(10))
    s.next_out, s.avail_out = C.addressof(obuf), 64
    assert lib.lzma_code(C.byref(s), 1) == 11  # LZMA_SYNC_FLUSH unsupported by the MT encoder -> LZMA_PROG_ERROR
    s.next_in, s.avail_in = C.addressof(ibuf), 10
    assert lib.lzma_code(C.byref(s), FINISH) in (0, 1)
    # changing the action (or avail_in) after LZMA_FINISH started is a programming error (common.c:253-281)
    assert lib.lzma_code(C.byref(s), RUN) == 11
    lib.lzma_end(C.byref(s))
    # reserved fields must be zero
    s2 = LzmaStream()
    assert lib.lzma_stream_encoder_mt(C.byref(s2), C.byref(m)) == 0
    s2.reserved_int2 = 1
    assert lib.lzma_code(C.byref(s2), RUN) == 8
    s2.reserved_int2 = 0
    lib.lzma_end(C.byref(s2))


def test_decoder_finishes_unsized_stream_under_lzma_run_only(lib):
    """Callers that never pass LZMA_FINISH (Python's lzma module, libarchive): the reference's decoder returns
    LZMA_STREAM_END under LZMA_RUN once the Stream Footer is in (stream_decoder.c:309-331).  Single-threaded encoders
    write Blocks without sizes, so the end of the Stream is only found by decoding; here the input arrives in 8 KiB
    pieces with LZMA_RUN throughout.  Also a ratio far above 64 : 1 (zeros), where the first output guess is too small.
    The Streams are the reference's `xz -6 -T1` output for these inputs (tests/golden/ref_xz_*_T1.xz)."""
    for name, data in (("T6_300000", bytes(X.gendata("T", 300000)[:300000])), ("zeros_40000000", bytes(40 * 1000 * 1000))):
        comp = open(os.path.join(GOLD, f"ref_xz_{name}_T1.xz"), "rb").read()
        d = LzmaStream()
        assert lib.lzma_stream_decoder(C.byref(d), C.c_uint64((1 << 64) - 1), C.c_uint32(0)) == 0
        ret, back = _drive(lib, d, comp, 8192, 1 << 20, final_action=RUN)
        lib.lzma_end(C.byref(d))
        assert ret == 1 and back == data


def test_decoder_buf_error_and_data_error_latching(lib):
    n = 40000
    buf = X.gendata("E", n)
    xz = X.oracle_encode(buf, n, 1, 1 << 14)
    d = LzmaStream()
    assert lib.lzma_stream_decoder(C.byref(d), C.c_uint64((1 << 64) - 1), C.c_uint32(0)) == 0
    ret, back = _drive(lib, d, xz[: len(xz) // 2], 4096, 1 << 16)  # truncated + LZMA_FINISH
    assert ret == 10  # LZMA_BUF_ERROR on the second call without progress
    lib.lzma_end(C.byref(d))
    bad = bytearray(xz); bad[len(xz) // 2] ^= 0x21
    d = LzmaStream()
    assert lib.lzma_stream_decoder(C.byref(d), C.c_uint64((1 << 64) - 1), C.c_uint32(0)) == 0
    ret, _ = _drive(lib, d, bytes(bad), 1 << 20, 1 << 20)
    assert ret == 9
    assert lib.lzma_code(C.byref(d), FINISH) == 11  # latched (common.c:368-372)
    lib.lzma_end(C.byref(d))
    # lzma_stream_decoder_mt entry point runs the same decoder
    m = LzmaMt(); m.threads = 8; m.memlimit_stop = (1 << 64) - 1; m.memlimit_threading = (1 << 64) - 1
    d = LzmaStream()
    assert lib.lzma_stream_decoder_mt(C.byref(d), C.byref(m)) == 0
    ret, back = _drive(lib, d, xz, 5000, 7000)
    assert ret == 1 and back == bytes(buf[:n])
    lib.lzma_end(C.byref(d))


def test_concatenated_streams_and_padding(lib):
    """LZMA_CONCATENATED (stream_decoder.c:334-371): corpus verdicts with the flag, plus two real Streams
    with 8 bytes of Stream Padding between them, and a bad (non multiple of 4) padding."""
    import hashlib, json, os
    gold = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    verdicts = json.load(open(os.path.join(gold, "decode_verdicts.json")))
    for name, v in sorted(verdicts.items()):   # (Delta / BCJ chains included: xzb_k_filter)
        data = open(os.path.join(gold, "ref_files", name), "rb").read()
        d = LzmaStream()
        assert lib.lzma_stream_decoder(C.byref(d), C.c_uint64((1 << 64) - 1), C.c_uint32(0x08)) == 0
        ret, out = _drive(lib, d, data, 1 << 20, 1 << 20)
        lib.lzma_end(C.byref(d))
        want = v["ret_concat"]
        assert (ret == 1 and want == 0) or ret == want, (name, ret, want)
        if want == 0:
            assert hashlib.sha256(out).hexdigest() == v["out_concat_sha256"], name
    a, b = X.gendata("T", 100000), X.gendata("E", 70000)
    xa, xb = X.oracle_encode(a, 100000, 6, 1 << 16), X.oracle_encode(b, 70000, 1, 1 << 15)
    assert [X.digest(xa), X.digest(xb)] == X.ref_golden()["concat_pad"]["inputs"]
    for pad, ok in ((0, True), (8, True), (6, False)):
        d = LzmaStream()
        assert lib.lzma_stream_decoder(C.byref(d), C.c_uint64((1 << 64) - 1), C.c_uint32(0x08)) == 0
        ret, out = _drive(lib, d, xa + b"\0" * pad + xb, 30000, 50000)
        lib.lzma_end(C.byref(d))
        if ok:
            assert ret == 1 and out == bytes(a[:100000]) + bytes(b[:70000])
        else:
            assert ret == 9
        assert (X.ref_golden()["concat_pad"][str(pad)] == 0) == ok   # the reference's verdict on the same bytes


# ---- one-shot buffer API: lzma_easy_buffer_encode / lzma_stream_buffer_encode / lzma_stream_buffer_decode ----
import hashlib
import json
import os
import sys

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
sys.path.insert(0, GOLD)


def _easy_buffer_encode(lib, data, n, preset, check, cap=None, start=0):
    lib.lzma_stream_buffer_bound.restype = C.c_size_t
    lib.lzma_stream_buffer_bound.argtypes = [C.c_size_t]
    cap = lib.lzma_stream_buffer_bound(n) + start if cap is None else cap
    out = (C.c_uint8 * max(cap, 1))()
    pos = C.c_size_t(start)
    r = lib.lzma_easy_buffer_encode(C.c_uint32(preset), C.c_int(check), None, data, C.c_size_t(n), out, C.byref(pos), C.c_size_t(cap))
    return r, bytes(out[start: pos.value]), pos.value


def _buffer_encode_cases():
    return json.load(open(os.path.join(GOLD, "buffer_golden.json")))["encode"]


@pytest.mark.parametrize("case", _buffer_encode_cases(), ids=lambda c: f"{c['kind']}-{c['preset']:#x}-{c['size']}-c{c['check']}")
def test_easy_buffer_encode_matches_reference_golden(lib, case):
    """Bytes of the reference's lzma_easy_buffer_encode (SHA-256 in tests/golden/buffer_golden.json);
    small cases are also compared byte by byte with the oracle's restatement."""
    n = case["size"]
    buf = X.gendata(case["kind"], n)
    r, out, _ = _easy_buffer_encode(lib, buf, n, case["preset"], case["check"])
    assert r == 0
    assert len(out) == case["xz_size"] and hashlib.sha256(out).hexdigest() == case["xz_sha256"]
    if n <= 65537:
        assert out == X.oracle_buffer_encode(buf, n, case["preset"], case["check"])


def test_stream_buffer_encode_filters_and_output_window(lib):
    from test_api_cpu import LzmaFilter, LzmaOptionsLzma
    n = 200000
    buf = X.gendata("T", n)
    o = LzmaOptionsLzma()
    assert lib.lzma_lzma_preset(C.byref(o), C.c_uint32(4)) == 0
    o.nice_len, o.depth, o.lc, o.lp = 48, 20, 2, 1
    f = (LzmaFilter * 2)()
    f[0].id, f[0].options = 0x21, C.cast(C.pointer(o), C.c_void_p)
    f[1].id = (1 << 64) - 1
    xo = X.preset_options(4); xo.nice_len, xo.depth, xo.lc, xo.lp = 48, 20, 2, 1
    want = X.oracle_buffer_encode(buf, n, 4, 1, opts=xo)
    cap = len(want) + 100
    out = (C.c_uint8 * cap)()
    pos = C.c_size_t(100)  # output lands at *out_pos, bytes before it stay untouched
    for i in range(100):
        out[i] = 0xEE
    assert lib.lzma_stream_buffer_encode(f, C.c_int(1), None, buf, C.c_size_t(n), out, C.byref(pos), C.c_size_t(cap)) == 0
    assert pos.value == cap and bytes(out[100:]) == want and bytes(out[:100]) == b"\xee" * 100
    # one byte short: LZMA_BUF_ERROR and *out_pos is unchanged (stream_buffer_encoder.c:62-66, 134-139)
    pos.value = 100
    assert lib.lzma_stream_buffer_encode(f, C.c_int(1), None, buf, C.c_size_t(n), out, C.byref(pos), C.c_size_t(cap - 1)) == 10
    assert pos.value == 100
    # a filter chain the GPU path does not take
    f[0].id = 0x03
    assert lib.lzma_stream_buffer_encode(f, C.c_int(1), None, buf, C.c_size_t(n), out, C.byref(pos), C.c_size_t(cap)) == 8
    # incompressible input takes the uncompressed-chunk fallback and still fits lzma_stream_buffer_bound
    rb = X.gendata("R", 70000)
    r, xz, _ = _easy_buffer_encode(lib, rb, 70000, 6, 4)
    assert r == 0 and xz == X.oracle_buffer_encode(rb, 70000, 6, 4)


def _buffer_decode_cases():
    import make_golden as MG
    g = json.load(open(os.path.join(GOLD, "buffer_golden.json")))["decode"]
    return [(name, kind, preset, n, m, g[name]) for name, kind, preset, n, m in MG.buffer_decode_cases()]


@pytest.mark.parametrize("name,kind,preset,n,m,want", _buffer_decode_cases(), ids=lambda v: v if isinstance(v, str) and "_" in v else None)
def test_stream_buffer_decode_matches_reference_verdicts(lib, name, kind, preset, n, m, want):
    """Return code, consumed input and produced output of the reference's lzma_stream_buffer_decode
    (common/stream_buffer_decoder.c:14-92) on good, truncated, corrupt, concatenated and too-small-output
    cases; the inputs are rebuilt from the generators and the oracle's (reference-identical) encoder."""
    import make_golden as MG
    data, cap, flags = MG.buffer_case_input(kind, preset, n, m, lambda b, nn, p, c: X.oracle_buffer_encode(b, nn, p, c))
    out = (C.c_uint8 * max(cap, 1))()
    ip, op = C.c_size_t(0), C.c_size_t(0)
    ml = C.c_uint64((1 << 64) - 1)
    r = lib.lzma_stream_buffer_decode(C.byref(ml), C.c_uint32(flags), None, data, C.byref(ip), C.c_size_t(len(data)), out, C.byref(op), C.c_size_t(cap))
    assert (r, ip.value, op.value) == (want["ret"], want["in_used"], want["out_size"]), name
    if r == 0:
        assert hashlib.sha256(bytes(out[: op.value])).hexdigest() == want["out_sha256"]


def test_buffer_roundtrip_through_reference_decoder(lib):
    """Cross-check in the other direction: our one-shot Stream is the reference's, and the reference's
    lzma_stream_buffer_decode gave the input back from it (tests/golden/ref_checks_golden.json)."""
    n = 3 * (1 << 20) + 17
    buf = X.gendata("E", n)
    r, xz, _ = _easy_buffer_encode(lib, buf, n, 2, 4)
    ref = X.ref_golden()["buffer_roundtrip"]
    assert r == 0 and X.digest(xz) == ref["xz"]
    assert ref["decode"] == [0, len(xz)] + X.digest(bytes(buf[:n]))


# ---- return-code sequences of the streaming decoder (LZMA_TELL_*, LZMA_CONCATENATED, LZMA_IGNORE_CHECK) ----
def _trace_cases():
    g = json.load(open(os.path.join(GOLD, "stream_trace_golden.json")))
    return sorted(g.items())


def _trace_inputs():
    import make_golden as MG
    d = {n: open(os.path.join(GOLD, "ref_files", n), "rb").read() for n in os.listdir(os.path.join(GOLD, "ref_files"))}
    d.update(MG.trace_inputs())
    return d


_TRACE_INPUTS = None


@pytest.mark.parametrize("key,want", _trace_cases(), ids=lambda v: v if isinstance(v, str) else None)
def test_stream_decoder_code_sequences_match_reference(lib, key, want):
    """lzma_stream_decoder(flags) + the lzma_code(LZMA_FINISH) loop of src/xz/coder.c: every return code
    other than LZMA_OK, with lzma_get_check() after it, equals the reference's sequence
    (tests/golden/stream_trace_golden.json), as do the bytes produced (CRC32, CRC64 and SHA-256 Streams)."""
    global _TRACE_INPUTS
    if _TRACE_INPUTS is None:
        _TRACE_INPUTS = _trace_inputs()
    name, fl = key.split("|")
    flags = int(fl, 16)
    data = _TRACE_INPUTS[name]
    lib.lzma_get_check.restype = C.c_int
    s = LzmaStream()
    # Every third case goes in through lzma_stream_decoder_mt (threads = 4, no limits): the reference's threaded decoder
    # gives exactly the recorded sequences and bytes for all 750 cases (tests/test_mt_traces_cpu.py checks that against
    # the unmodified reference), so the same golden file pins both entry points.
    if sum(key.encode()) % 3 == 0:
        m = LzmaMt(); m.flags = flags; m.threads = 4; m.memlimit_stop = (1 << 64) - 1; m.memlimit_threading = (1 << 64) - 1
        assert lib.lzma_stream_decoder_mt(C.byref(s), C.byref(m)) == 0
    else:
        assert lib.lzma_stream_decoder(C.byref(s), C.c_uint64((1 << 64) - 1), C.c_uint32(flags)) == 0
    cap = 1 << 22
    obuf = (C.c_uint8 * cap)()
    ibuf = (C.c_uint8 * max(len(data), 1)).from_buffer_copy(data or b"\0")
    s.next_in, s.avail_in, s.next_out, s.avail_out = C.addressof(ibuf), len(data), C.addressof(obuf), cap
    codes = []
    for _ in range(100):
        ret = lib.lzma_code(C.byref(s), FINISH)
        if ret == 0:
            continue
        codes.append([ret, lib.lzma_get_check(C.byref(s))])
        if ret in (2, 3, 4):
            continue
        break
    out = bytes(obuf[: s.total_out])
    lib.lzma_end(C.byref(s))
    exp = [list(c) for c in want["codes"]]
    exp_size, exp_sha = want["out_size"], want["out_sha256"]
    # (files with Delta / BCJ filters in front of LZMA2 go through xzb_k_filter and must match like the rest)
    # lzma_get_check() after an error code is whatever the coder last stored (uninitialised when the
    # Stream Header itself was bad): compare it only for LZMA_STREAM_END and the LZMA_TELL_* codes
    norm = lambda cs: [c if c[0] <= 4 else [c[0], None] for c in cs]
    assert norm(codes) == norm(exp), (key, codes, exp)
    assert len(out) == exp_size and hashlib.sha256(out).hexdigest() == exp_sha


def _block_cases():
    return json.load(open(os.path.join(GOLD, "buffer_golden.json")))["block_buffer_encode"]


@pytest.mark.parametrize("g", _block_cases(), ids=lambda c: f"{c['kind']}-{c['preset']:#x}-{c['size']}-c{c['check']}")
def test_block_buffer_encode_matches_reference_golden(lib, g):
    """lzma_block_buffer_encode: Block bytes, header_size, compressed_size and raw_check of the reference
    (tests/golden/buffer_golden.json), including the uncompressed-chunk fallback on random input."""
    from test_api_cpu import LzmaBlock, LzmaFilter, LzmaOptionsLzma
    n = g["size"]
    buf = X.gendata(g["kind"], n)
    o = LzmaOptionsLzma()
    assert lib.lzma_lzma_preset(C.byref(o), C.c_uint32(g["preset"])) == 0
    f = (LzmaFilter * 2)()
    f[0].id, f[0].options = 0x21, C.cast(C.pointer(o), C.c_void_p)
    f[1].id = (1 << 64) - 1
    lib.lzma_block_buffer_bound.restype = C.c_size_t
    lib.lzma_block_buffer_bound.argtypes = [C.c_size_t]
    cap = lib.lzma_block_buffer_bound(n) + 7
    out = (C.c_uint8 * cap)()
    b = LzmaBlock(); b.check, b.filters = g["check"], C.cast(f, C.c_void_p)
    pos = C.c_size_t(3)
    assert lib.lzma_block_buffer_encode(C.byref(b), None, buf, C.c_size_t(n), out, C.byref(pos), C.c_size_t(cap)) == 0
    blk = bytes(out[3: pos.value])
    assert len(blk) == g["block_size"] and hashlib.sha256(blk).hexdigest() == g["block_sha256"]
    assert (b.header_size, b.compressed_size, b.uncompressed_size) == (g["header_size"], g["compressed_size"], n)
    cs = {0: 0, 1: 4, 4: 8, 10: 32}[g["check"]]
    assert bytes(b.raw_check)[:cs].hex() == g["raw_check"][: 2 * cs]
    if n > 0:  # one byte short of what it needs: LZMA_BUF_ERROR, *out_pos untouched
        pos = C.c_size_t(0)
        assert lib.lzma_block_buffer_encode(C.byref(b), None, buf, C.c_size_t(n), out, C.byref(pos), C.c_size_t(g["block_size"] - 1)) == 10
        assert pos.value == 0


def _memlimit_cases():
    return sorted(json.load(open(os.path.join(GOLD, "memlimit_trace_golden.json"))).items())


@pytest.mark.parametrize("key,want", _memlimit_cases(), ids=lambda v: v if isinstance(v, str) else None)
def test_stream_decoder_memlimit_sequences_match_reference(lib, key, want):
    """lzma_stream_decoder(memlimit): LZMA_MEMLIMIT_ERROR at the first Block that would need more (with the
    reference's figure from lzma_memusage), lzma_memlimit_set() below / at that figure, decoding goes on
    (stream_decoder.c:199-232, 389-408; caller pattern src/xz/coder.c:1292-1316)."""
    global _TRACE_INPUTS
    if _TRACE_INPUTS is None:
        _TRACE_INPUTS = _trace_inputs()
    name, fl, ml = key.split("|")
    flags, memlimit = int(fl, 16), int(ml)
    data = _TRACE_INPUTS[name]
    lib.lzma_get_check.restype = C.c_int
    lib.lzma_memusage.restype = C.c_uint64
    lib.lzma_memlimit_get.restype = C.c_uint64
    s = LzmaStream()
    assert lib.lzma_stream_decoder(C.byref(s), C.c_uint64(memlimit), C.c_uint32(flags)) == 0
    assert lib.lzma_memlimit_get(C.byref(s)) == max(memlimit, 1)
    cap = 1 << 22
    obuf = (C.c_uint8 * cap)()
    ibuf = (C.c_uint8 * max(len(data), 1)).from_buffer_copy(data or b"\0")
    s.next_in, s.avail_in, s.next_out, s.avail_out = C.addressof(ibuf), len(data), C.addressof(obuf), cap
    codes, seen = [], 0
    for _ in range(100):
        ret = lib.lzma_code(C.byref(s), FINISH)
        if ret == 0:
            continue
        codes.append(ret | (lib.lzma_get_check(C.byref(s)) << 8))
        if ret in (2, 3, 4):
            continue
        if ret == 6 and seen == 0:
            seen = lib.lzma_memusage(C.byref(s))
            low = lib.lzma_memlimit_set(C.byref(s), C.c_uint64(seen - 1))
            ok = lib.lzma_memlimit_set(C.byref(s), C.c_uint64(seen))
            codes.append(0x8000 | low | (ok << 8))
            if ok == 0:
                continue
        break
    if seen == 0:
        seen = lib.lzma_memusage(C.byref(s))
    out = bytes(obuf[: s.total_out])
    lib.lzma_end(C.byref(s))
    norm = lambda cs: [c if (c & 0xFF) <= 6 or c & 0x8000 else c & 0xFF for c in cs]
    assert norm(codes) == norm(want["codes"]), (key, [hex(c) for c in codes], [hex(c) for c in want["codes"]])
    assert seen == want["memusage"] and len(out) == want["out_size"] and hashlib.sha256(out).hexdigest() == want["out_sha256"]


def test_stream_decoder_hands_over_complete_blocks_while_input_arrives(lib):
    """A long Stream is not buffered whole: every 64 complete Blocks are decoded as a part and cut out of the input
    buffer, their Index records kept for the check of the real Index at the end (xzb_stream_decode_prior).
    Output therefore appears while input is still arriving, the bytes and the final verdict are the same, and
    a corrupt Index entry / a corrupt late Block are still caught."""
    n, bs = 200 * 16384 + 777, 16384
    buf = X.gendata("T", n)
    data = bytes(buf[:n])
    xz = X.oracle_encode(buf, n, 1, bs)

    def run(stream, flags=0):
        s = LzmaStream()
        assert lib.lzma_stream_decoder(C.byref(s), C.c_uint64((1 << 64) - 1), C.c_uint32(flags)) == 0
        ibuf = (C.c_uint8 * len(stream)).from_buffer_copy(stream)
        obuf = (C.c_uint8 * (1 << 16))()
        out = bytearray()
        pos, first_out_at, ret = 0, None, 0
        s.next_out, s.avail_out = C.addressof(obuf), len(obuf)
        for _ in range(1_000_000):
            if s.avail_in == 0 and pos < len(stream):
                k = min(50000, len(stream) - pos)
                s.next_in, s.avail_in = C.addressof(ibuf) + pos, k
                pos += k
            ret = lib.lzma_code(C.byref(s), FINISH if pos == len(stream) else RUN)
            got = len(obuf) - s.avail_out
            if got:
                if first_out_at is None:
                    first_out_at = pos
                out += bytes(obuf[:got])
                s.next_out, s.avail_out = C.addressof(obuf), len(obuf)
            if ret != 0:
                break
        lib.lzma_end(C.byref(s))
        return ret, bytes(out), first_out_at

    ret, out, first_out_at = run(xz)
    assert ret == 1 and out == data
    assert first_out_at is not None and first_out_at < len(xz) * 2 // 3  # output before the last third of the input was fed
    ret, out, _ = run(xz + bytes(4) + xz, flags=0x08)  # two Streams, parts in both
    assert ret == 1 and out == data + data
    # a wrong byte in the LAST Block's data: every earlier Block is delivered intact (plus whatever the bad Block
    # decoded to before the error showed, as with the reference), then LZMA_DATA_ERROR
    idx_size = (int.from_bytes(xz[-8:-4], "little") + 1) * 4
    bad = bytearray(xz); bad[len(xz) - 12 - idx_size - 40] ^= 0x10
    ret, out, _ = run(bytes(bad))
    assert ret == 9 and len(out) >= 200 * bs and out[: 200 * bs] == data[: 200 * bs]
    # a wrong Index record of an early Block (already handed over): caught when the real Index is read
    bad = bytearray(xz); bad[len(xz) - 12 - idx_size + 3] ^= 0x01
    ret, out, _ = run(bytes(bad))
    assert ret == 9 and out == data


def test_misaligned_bcj_start_offset_fails_in_lzma_code_like_the_reference(lib):
    """A BCJ start offset that is not a multiple of the filter's alignment passes lzma_stream_encoder_mt (the chain is
    only validated by lzma_raw_encoder_memusage there) and comes back as LZMA_OPTIONS_ERROR from the first lzma_code,
    after the Stream Header, when a worker sets up its Block coder (simple_coder.c:276-278)."""
    from test_api_cpu import _chain, _mt
    keep = []
    arr = _chain([(0x07, 2), (0x21, 0)], keep)
    m = _mt(filters=C.cast(arr, C.c_void_p), threads=2)
    s = LzmaStream()
    assert lib.lzma_stream_encoder_mt(C.byref(s), C.byref(m)) == 0
    data = (C.c_uint8 * 100000)(); out = (C.c_uint8 * 200000)()
    s.next_in, s.avail_in, s.next_out, s.avail_out = C.addressof(data), 100000, C.addressof(out), 200000
    assert lib.lzma_code(C.byref(s), FINISH) == 8
    assert s.total_in == 100000 and s.total_out == 12
    assert lib.lzma_code(C.byref(s), FINISH) == 11   # latched (common.c:368-372)
    lib.lzma_end(C.byref(s))
