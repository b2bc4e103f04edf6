"""Delta / BCJ filters (xz_b200/csrc/xzb_filters.cuh, compiled for the host by tests/hostsim) against the unmodified
reference: the bytes the reference's filter chain hands to its LZMA2 encoder (raw encoder with the chain, raw decoder
with LZMA2 alone) and the inverse direction, on inputs built to trigger each filter's conversions.  The reference's
output on these inputs is recorded as SHA-256 in tests/golden/ref_checks_golden.json."""
import ctypes as C
import hashlib
import os
import random

import pytest

import xzlibs as X

HS = os.path.join(X.ROOT, "tests", "hostsim", "libhostsim.so")

DELTA, X86, POWERPC, IA64, ARM, ARMTHUMB, SPARC, ARM64, RISCV = 3, 4, 5, 6, 7, 8, 9, 10, 11
BCJ_CASES = [(X86, 0), (X86, 4096), (ARM, 0), (ARM, 8), (ARMTHUMB, 0), (ARMTHUMB, 2), (POWERPC, 0), (POWERPC, 64),
             (SPARC, 0), (SPARC, 4), (ARM64, 0), (ARM64, 0x10000), (IA64, 0), (IA64, 32), (RISCV, 0), (RISCV, 0x1002)]
BCJ_SIZES = [0, 1, 3, 4, 5, 15, 16, 17, 1000, 65537]
DELTA_DISTS = [1, 2, 3, 4, 255, 256]
DELTA_SIZES = [0, 1, 2, 255, 256, 257, 70001]


def sha(b):
    return hashlib.sha256(b).hexdigest()


def ours(fid, arg, enc, data):
    lib = C.CDLL(HS)
    buf = (C.c_uint8 * len(data)).from_buffer_copy(bytes(data))
    lib.hostsim_filter_apply(C.c_uint32(fid), C.c_uint32(arg), C.c_int(enc), buf, C.c_uint32(len(data)))
    return bytes(buf)


def codeish(fid, n, seed):
    """Random bytes salted with the opcode patterns the filter looks for (so conversions really happen)."""
    rnd = random.Random(seed)
    b = bytearray(rnd.getrandbits(8) for _ in range(n))
    for _ in range(n // 12 if n >= 64 else 0):
        i = rnd.randrange(0, n - 32)
        if fid == X86:
            b[i] = rnd.choice((0xE8, 0xE9)); b[i + 4] = rnd.choice((0x00, 0xFF))
            if rnd.random() < 0.3 and i + 9 < n:
                b[i + 5] = 0xE8; b[i + 9] = rnd.choice((0x00, 0xFF))   # back-to-back calls exercise prev_mask
        elif fid == ARM:
            i &= ~3; b[i + 3] = 0xEB
        elif fid == ARMTHUMB:
            i &= ~1; b[i + 1] = 0xF0 | rnd.getrandbits(3); b[i + 3] = 0xF8 | rnd.getrandbits(3)
        elif fid == POWERPC:
            i &= ~3; b[i] = 0x48 | rnd.getrandbits(2); b[i + 3] = (b[i + 3] & 0xFC) | 1
        elif fid == SPARC:
            i &= ~3
            if rnd.random() < 0.5: b[i] = 0x40; b[i + 1] &= 0x3F
            else: b[i] = 0x7F; b[i + 1] |= 0xC0
        elif fid == ARM64:
            i &= ~3
            if rnd.random() < 0.5: b[i + 3] = 0x94 | rnd.getrandbits(2)
            else: b[i + 3] = 0x90 | (rnd.getrandbits(2) << 5); b[i + 2] = rnd.choice((0x00, 0x01, 0xFE, 0xFF)); 
        elif fid == RISCV:
            i &= ~1
            k = rnd.random()
            if k < 0.35:      # JAL x1 / x5
                b[i] = 0xEF; b[i + 1] = (b[i + 1] & 0xF0) | rnd.choice((0x00, 0x02))
            elif k < 0.8:     # AUIPC rd, then an I-type instruction with rs1 = rd
                rd = rnd.choice((1, 3, 5, 6, 10, 17, 31))
                w = (rnd.getrandbits(20) << 12) | (rd << 7) | 0x17
                b[i:i + 4] = w.to_bytes(4, "little")
                w2 = (rnd.getrandbits(12) << 20) | (rd << 15) | (rnd.getrandbits(3) << 12) | (rnd.getrandbits(5) << 7) | rnd.choice((0x03, 0x13, 0x67))
                b[i + 4:i + 8] = w2.to_bytes(4, "little")
            else:             # AUIPC with rd = x0 / x2 (the forms the encoder has to escape)
                w = (rnd.getrandbits(20) << 12) | (rnd.choice((0, 2)) << 7) | 0x17
                b[i:i + 4] = w.to_bytes(4, "little")
        elif fid == IA64:
            i &= ~15; b[i] = (b[i] & 0xE0) | rnd.choice((16, 17, 18, 19, 22, 23, 24, 25, 28, 29))
            for s in (5, 46, 87):   # opcode 5 in bits 37..40 of a slot, btype 0 in bits 6..8... set some bits to make matches likely
                bp = s + 37
                for k in range(4):
                    byte, bit = (bp + k) >> 3, (bp + k) & 7
                    if (0x5 >> k) & 1: b[i + byte] |= 1 << bit
                    else: b[i + byte] &= ~(1 << bit)
                for k in range(3):
                    byte, bit = (s + 9 + k) >> 3, (s + 9 + k) & 7
                    b[i + byte] &= ~(1 << bit)
    return bytes(b)


@pytest.mark.parametrize("fid,arg", BCJ_CASES)
@pytest.mark.parametrize("n", BCJ_SIZES)
def test_bcj_matches_reference_both_directions(fid, arg, n):
    data = codeish(fid, n, 1000 * fid + n)
    ref_enc, ref_dec = X.ref_golden()["bcj"][f"{fid}|{arg}|{n}"]
    enc = ours(fid, arg, 1, data)
    assert sha(enc) == ref_enc
    assert ours(fid, arg, 0, enc) == data
    # decoding arbitrary bytes (not produced by the encoder) must also agree
    assert sha(ours(fid, arg, 0, data)) == ref_dec
    if n >= 1000:
        assert enc != data   # the salted patterns did convert something


@pytest.mark.parametrize("dist", DELTA_DISTS)
@pytest.mark.parametrize("n", DELTA_SIZES)
def test_delta_matches_reference_both_directions(dist, n):
    rnd = random.Random(dist * 7 + n)
    data = bytes(rnd.getrandbits(8) for _ in range(n))
    ref_enc, ref_dec = X.ref_golden()["delta"][f"{dist}|{n}"]
    enc = ours(DELTA, dist, 1, data)
    assert sha(enc) == ref_enc
    assert ours(DELTA, dist, 0, enc) == data
    assert sha(ours(DELTA, dist, 0, data)) == ref_dec
