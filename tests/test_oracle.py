"""CPU tests (-m "not gpu"): pin the oracle (oracle/liboracle.so) against
  * the reference's own golden vectors / KATs / decoder corpus (tests/golden/), and
  * what the unmodified reference produced on the same inputs (tests/golden/ref_checks_golden.json).
"""
import ctypes as C
import glob
import hashlib
import json
import os

import pytest

import xzlibs as X

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
MiB = 1 << 20


def test_crc_kats():
    kat = json.load(open(os.path.join(GOLD, "kat.json")))
    o = X.oracle()
    assert o.xzo_crc32(b"123456789", 9, 0) == kat["crc32_123456789"] == kat["ref_crc32_123456789"]
    assert o.xzo_crc64(b"123456789", 9, 0) == kat["crc64_123456789"] == kat["ref_crc64_123456789"]
    # split/unaligned variants, like tests/test_check.c:56-110
    c = 0
    for ch in b"123456789":
        c = o.xzo_crc32(bytes([ch]), 1, c)
    assert c == kat["crc32_123456789"]
    c = o.xzo_crc64(b"1234", 4, 0)
    assert o.xzo_crc64(b"56789", 5, c) == kat["crc64_123456789"]


def test_microlzma_encoder_kat():
    """The only encoder-output KAT in the reference tree (tests/test_microlzma.c:20-32)."""
    kat = json.load(open(os.path.join(GOLD, "kat.json")))
    o = X.preset_options(6)
    out = (C.c_uint8 * 65536)()
    sz = C.c_size_t()
    data = b"Hello\nWorld\n"
    assert X.oracle().xzo_microlzma_encode(data, C.c_size_t(len(data)), C.byref(o), out, C.c_size_t(65536), C.byref(sz)) == 0
    assert sz.value == 17
    assert X.oracle().xzo_crc32(bytes(out[:17]), 17, 0) == kat["microlzma_hello_world_crc32"]


def _golden_cases(max_size):
    cases = json.load(open(os.path.join(GOLD, "encode_golden.json")))
    return [c for c in cases if c["size"] <= max_size]


@pytest.mark.parametrize("case", _golden_cases(4 * MiB), ids=lambda c: f"{c['kind']}-{c['preset']:#x}-{c['size']}-{c['block_size']}")
def test_oracle_encoder_matches_reference_golden(case):
    buf = X.gendata(case["kind"], case["size"])
    out = X.oracle_encode(buf, case["size"], case["preset"], case["block_size"], case["check"])
    assert len(out) == case["xz_size"]
    assert hashlib.sha256(out).hexdigest() == case["xz_sha256"]
    r, back = X.oracle_decode(out, case["size"])
    assert r == 0 and back == bytes(buf[: case["size"]])


def _buffer_cases():
    g = json.load(open(os.path.join(GOLD, "buffer_golden.json")))["encode"]
    return [c for c in g if c["size"] <= 300000 or (c["size"] <= 4 * MiB and c["preset"] in (0, 3))]


@pytest.mark.parametrize("case", _buffer_cases(), ids=lambda c: f"{c['kind']}-{c['preset']:#x}-{c['size']}-c{c['check']}")
def test_oracle_buffer_encoder_matches_reference_golden(case):
    """xzo_stream_buffer_encode == the reference's lzma_easy_buffer_encode (one Block,
    lzma_block_buffer_encode framing): SHA-256 from tests/golden/buffer_golden.json."""
    buf = X.gendata(case["kind"], case["size"])
    out = X.oracle_buffer_encode(buf, case["size"], case["preset"], case["check"])
    assert len(out) == case["xz_size"] and hashlib.sha256(out).hexdigest() == case["xz_sha256"]


def test_oracle_buffer_encoder_vs_live_reference():
    gold = X.ref_golden()["buffer_encode"]
    for kind, preset, n in (("T", 6, 1234567), ("E", 9 | X.XZ_PRESET_EXTREME, 200001), ("R", 1, 131072), ("L", 3, 700000)):
        buf = X.gendata(kind, n)
        for check in (0, 1, 4):
            assert X.digest(X.oracle_buffer_encode(buf, n, preset, check)) == gold[f"{kind}|{preset:#x}|{n}|{check}"]


def test_oracle_encoder_config0_full_size():
    """BASELINE.json configs[0]: xz -1, 16 MiB synthetic text, one 16 MiB block (CPU plumbing)."""
    case = [c for c in json.load(open(os.path.join(GOLD, "encode_golden.json")))
            if c["kind"] == "T" and c["preset"] == 1 and c["size"] == 16 * MiB][0]
    buf = X.gendata("T", case["size"])
    cnt = X.Counters()
    out = X.oracle_encode(buf, case["size"], 1, case["block_size"], counters=cnt)
    assert hashlib.sha256(out).hexdigest() == case["xz_sha256"]
    assert cnt.n_raw_with_read_ahead == 0 or cnt.n_chunks_raw > 0


def test_decoder_corpus_verdicts():
    """tests/files/*.xz of the reference: same verdict (lzma_ret) and same bytes as the reference."""
    verdicts = json.load(open(os.path.join(GOLD, "decode_verdicts.json")))
    out_of_scope = ("delta", "arm64", "bcj")  # non-LZMA2 filters: SURVEY section 2 rows 23, 24
    n = 0
    for name, v in sorted(verdicts.items()):
        if any(t in name for t in out_of_scope):
            continue
        data = open(os.path.join(GOLD, "ref_files", name), "rb").read()
        r, out = X.oracle_decode(data, 1 << 22)
        assert r == v["ret"], (name, r, v["ret"])
        if r == 0:
            assert len(out) == v["out_size"] and hashlib.sha256(out).hexdigest() == v["out_sha256"], name
        n += 1
    assert n > 50


@pytest.mark.parametrize("kind", "TER")
def test_oracle_vs_live_reference(kind):
    """Same inputs: oracle restatement == unmodified reference, encode, and the reference's decoders (single- and
    multi-threaded) give the input back from that Stream."""
    for preset, n, bs in ((1, 1 * MiB + 3, 512 * 1024), (6, 600001, 256 * 1024), (3, 700000, 1 * MiB)):
        buf = X.gendata(kind, n)
        a = X.oracle_encode(buf, n, preset, bs)
        ref = X.ref_golden()["stream_encode"][f"{kind}|{preset}|{n}|{bs}"]
        assert X.digest(a) == ref["xz"]
        want = [0] + X.digest(bytes(buf[:n]))
        assert ref["decode"] == want and ref["decode_mt"] == want


def test_oracle_vs_live_reference_all_match_finders():
    buf = X.gendata("T", 300000)
    gold = X.ref_golden()["match_finders"]
    for mode in (1, 2):
        for mf in (0x03, 0x04, 0x12, 0x13, 0x14):
            for lc, lp, pb in ((3, 0, 2), (0, 2, 0), (4, 0, 4), (1, 3, 1)):
                o = X.LzmaOptions(1 << 20, lc, lp, pb, mode, 32, mf, 0)
                assert X.digest(X.oracle_encode(buf, 300000, 0, 1 << 20, opts=o)) == gold[f"{mode}|{mf:#x}|{lc}|{lp}|{pb}"]


def test_truncated_and_corrupt_streams():
    buf = X.gendata("T", 50000)
    xz = X.oracle_encode(buf, 50000, 6, 1 << 16)
    for cut in (0, 5, 11, 12, 13, 40, len(xz) // 2, len(xz) - 1):
        r, _ = X.oracle_decode(xz[:cut], 50000)
        assert r == 10, (cut, r)  # LZMA_BUF_ERROR
    bad = bytearray(xz)
    bad[len(xz) // 2] ^= 0x55
    r, _ = X.oracle_decode(bytes(bad), 50000)
    assert r == 9
    ref = X.ref_golden()["truncated"]
    assert X.digest(xz) == ref["xz"]
    for cut in (5, 40, len(xz) // 2, len(xz) - 1):
        assert ref["cut"][str(cut)] == 10
    assert ref["flipped"] == 9
