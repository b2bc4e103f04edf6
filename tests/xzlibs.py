"""ctypes bindings used by the tests: the oracle (checker), oracle/_ref (the unmodified
reference, when built), the input generator, and the product C-ABI library."""
import ctypes as C
import hashlib
import json
import os

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
XZ_PRESET_EXTREME = 0x80000000
CHECK_NONE, CHECK_CRC32, CHECK_CRC64 = 0, 1, 4


class LzmaOptions(C.Structure):
    _fields_ = [(n, C.c_uint32) for n in ("dict_size", "lc", "lp", "pb", "mode", "nice_len", "mf", "depth")]


class Counters(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("n_pos", "n_nodes", "n_cmp_bytes", "n_pairs", "n_symbols",
                                          "n_chunks_lzma", "n_chunks_raw", "n_raw_with_read_ahead")]


_cache = {}


def _load(path):
    if path not in _cache:
        _cache[path] = C.CDLL(path)
    return _cache[path]


def oracle():
    lib = _load(os.path.join(ROOT, "oracle", "liboracle.so"))
    lib.xzo_stream_bound.restype = C.c_size_t
    lib.xzo_stream_bound.argtypes = [C.c_size_t, C.c_uint64]
    lib.xzo_block_bound.restype = C.c_uint64
    lib.xzo_block_bound.argtypes = [C.c_uint64]
    lib.xzo_crc32.restype = C.c_uint32
    lib.xzo_crc32.argtypes = [C.c_char_p, C.c_size_t, C.c_uint32]
    lib.xzo_crc64.restype = C.c_uint64
    lib.xzo_crc64.argtypes = [C.c_char_p, C.c_size_t, C.c_uint64]
    lib.xzo_mf_dump.restype = C.c_uint64
    return lib


def have_ref():
    return os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libref_shim.so"))


def ref():
    lib = _load(os.path.join(ROOT, "oracle", "_ref", "libref_shim.so"))
    lib.ref_crc32.restype = C.c_uint32
    lib.ref_crc32.argtypes = [C.c_char_p, C.c_size_t, C.c_uint32]
    lib.ref_crc64.restype = C.c_uint64
    lib.ref_crc64.argtypes = [C.c_char_p, C.c_size_t, C.c_uint64]
    lib.ref_cputhreads.restype = C.c_uint32
    return lib


def gen():
    return _load(os.path.join(ROOT, "xz_b200", "libxzgen.so"))


def gendata(kind, n, off=0):
    """n bytes [off, off+n) of synthetic stream `kind` ('T','E','R','L') as a ctypes array."""
    b = (C.c_uint8 * max(n, 1))()
    assert gen().xzgen_fill(C.c_char(kind.encode()), b, C.c_size_t(n), C.c_uint64(off)) == 0
    return b


def preset_options(preset):
    o = LzmaOptions()
    assert oracle().xzo_lzma_preset(C.byref(o), C.c_uint32(preset)) == 0
    return o


def oracle_encode(buf, n, preset, block_size, check=CHECK_CRC64, opts=None, counters=None):
    lib = oracle()
    o = opts if opts is not None else preset_options(preset)
    cap = lib.xzo_stream_bound(n, block_size)
    out = (C.c_uint8 * cap)()
    sz = C.c_size_t()
    r = lib.xzo_stream_encode(buf, C.c_size_t(n), C.byref(o), C.c_uint32(check), C.c_uint64(block_size), out,
                              C.c_size_t(cap), C.byref(sz), C.byref(counters) if counters is not None else None)
    assert r == 0, r
    return bytes(out[:sz.value])


def oracle_buffer_encode(buf, n, preset, check=CHECK_CRC64, opts=None):
    """xzo_stream_buffer_encode: the restatement of lzma_stream_buffer_encode / lzma_easy_buffer_encode."""
    lib = oracle()
    lib.xzo_stream_buffer_bound.restype = C.c_size_t
    lib.xzo_stream_buffer_bound.argtypes = [C.c_size_t]
    o = opts if opts is not None else preset_options(preset)
    cap = lib.xzo_stream_buffer_bound(n)
    out = (C.c_uint8 * cap)()
    sz = C.c_size_t()
    r = lib.xzo_stream_buffer_encode(buf, C.c_size_t(n), C.byref(o), C.c_uint32(check), out, C.c_size_t(cap), C.byref(sz))
    assert r == 0, r
    return bytes(out[:sz.value])


def ref_buffer_encode(buf, n, preset, check=CHECK_CRC64):
    """lzma_easy_buffer_encode of the unmodified reference (oracle/_ref)."""
    r_ = ref()
    r_.ref_stream_buffer_bound.restype = C.c_size_t
    r_.ref_stream_buffer_bound.argtypes = [C.c_size_t]
    cap = r_.ref_stream_buffer_bound(n)
    out = (C.c_uint8 * cap)()
    sz = C.c_size_t()
    r = r_.ref_easy_buffer_encode(buf, C.c_size_t(n), C.c_uint32(preset), C.c_uint32(check), out, C.c_size_t(cap), C.byref(sz))
    assert r == 0, r
    return bytes(out[:sz.value])


def ref_block_buffer_encode(buf, n, preset, check=CHECK_CRC64):
    """lzma_block_buffer_encode of the unmodified reference: (block bytes, header_size, compressed_size, raw_check)."""
    cap = oracle().xzo_block_bound(n) + 64
    out = (C.c_uint8 * cap)(); sz = C.c_size_t(); hs = C.c_uint32(); cs = C.c_uint64(); us = C.c_uint64(); rc = (C.c_uint8 * 64)()
    r = ref().ref_block_buffer_encode(buf, C.c_size_t(n), C.c_uint32(preset), C.c_uint32(check), out, C.c_size_t(cap), C.byref(sz),
                                      C.byref(hs), C.byref(cs), C.byref(us), rc)
    assert r == 0 and us.value == n, r
    return bytes(out[: sz.value]), hs.value, cs.value, bytes(rc)


def ref_buffer_decode(data, cap, flags=0):
    """lzma_stream_buffer_decode of the unmodified reference: (ret, bytes, in_used)."""
    out = (C.c_uint8 * max(cap, 1))()
    used = C.c_size_t(); sz = C.c_size_t()
    r = ref().ref_stream_buffer_decode(data, C.c_size_t(len(data)), C.c_uint32(flags), out, C.c_size_t(cap), C.byref(used), C.byref(sz))
    return r, bytes(out[:sz.value]), used.value


def oracle_decode(data, cap):
    out = (C.c_uint8 * max(cap, 1))()
    sz = C.c_size_t()
    r = oracle().xzo_stream_decode(data, C.c_size_t(len(data)), out, C.c_size_t(cap), C.byref(sz))
    return r, bytes(out[:sz.value])


def ref_encode(buf, n, preset, block_size, check=CHECK_CRC64, threads=0, opts=None):
    cap = oracle().xzo_stream_bound(n, block_size)
    out = (C.c_uint8 * cap)()
    sz = C.c_size_t()
    if opts is None:
        r = ref().ref_encode_mt(buf, C.c_size_t(n), C.c_uint32(preset), C.c_uint64(block_size), C.c_uint32(check),
                                C.c_uint32(threads), out, C.c_size_t(cap), C.byref(sz))
    else:
        o = opts
        r = ref().ref_encode_mt_opts(buf, C.c_size_t(n), o.dict_size, o.lc, o.lp, o.pb, o.mode, o.nice_len, o.mf,
                                     o.depth, C.c_uint64(block_size), C.c_uint32(check), C.c_uint32(threads), out,
                                     C.c_size_t(cap), C.byref(sz))
    assert r == 0, r
    return bytes(out[:sz.value])


def ref_filter_apply(fid, arg, enc, data):
    """One Delta / BCJ filter of the unmodified reference over `data` (encoder direction when enc)."""
    n = len(data)
    out = (C.c_uint8 * n)()
    ids = (C.c_uint32 * 1)(fid); args = (C.c_uint32 * 1)(arg)
    r = ref().ref_filter_apply(ids, args, C.c_uint32(1), C.c_int(enc), bytes(data), C.c_size_t(n), out)
    assert r == 0, r
    return bytes(out)


def ref_chain_encode(data, chain, preset, bs, check=CHECK_CRC64):
    """lzma_stream_encoder_mt of the unmodified reference with the filter chain [(id, arg), ...] in front of LZMA2."""
    n = len(data)
    cap = n + n // 2 + 65536
    out = (C.c_uint8 * cap)()
    sz = C.c_size_t()
    ids = (C.c_uint32 * len(chain))(*[c[0] for c in chain])
    args = (C.c_uint32 * len(chain))(*[c[1] for c in chain])
    r = ref().ref_encode_mt_chain(data, C.c_size_t(n), ids, args, C.c_uint32(len(chain)), C.c_uint32(preset), C.c_uint64(bs), C.c_uint32(check),
                                  C.c_uint32(4), out, C.c_size_t(cap), C.byref(sz))
    assert r == 0, r
    return bytes(out[:sz.value])


def ref_golden():
    """What the tests compare with the reference on their own inputs (tests/golden/make_golden.py live)."""
    if "golden" not in _cache:
        with open(os.path.join(ROOT, "tests", "golden", "ref_checks_golden.json")) as f:
            _cache["golden"] = json.load(f)
    return _cache["golden"]


def digest(b):
    """[size, SHA-256] as ref_checks_golden.json stores the reference's output."""
    return [len(b), hashlib.sha256(b).hexdigest()]


def ref_decode(data, cap, mt=False):
    out = (C.c_uint8 * max(cap, 1))()
    sz = C.c_size_t()
    if mt:
        r = ref().ref_decode_mt(data, C.c_size_t(len(data)), C.c_uint32(0), out, C.c_size_t(cap), C.byref(sz))
    else:
        r = ref().ref_decode(data, C.c_size_t(len(data)), out, C.c_size_t(cap), C.byref(sz))
    return r, bytes(out[:sz.value])
