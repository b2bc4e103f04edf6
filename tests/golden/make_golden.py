#!/usr/bin/env python
"""Regenerates tests/golden/ from the UNMODIFIED reference (run in the build container only).

1. Copies the reference's own decoder fixtures for the LZMA2 path
   (/root/reference/tests/files/{good,bad,unsupported}-*.xz; semantics in tests/files/README:44-176)
   into tests/golden/ref_files/ and records the reference's verdict (lzma_ret of
   lzma_stream_decoder + lzma_code(FINISH), SHA-256 of the output) in decode_verdicts.json.
2. Runs the reference encoder (lzma_stream_encoder_mt via oracle/_ref) on seeded synthetic
   inputs and records SHA-256 + size of the .xz it produces in encode_golden.json.
   The inputs are regenerated from xz_b200/csrc/xzgen.c, so only hashes are stored.
4. (`make_golden.py buffer`) runs the reference's one-shot buffer API (lzma_easy_buffer_encode,
   lzma_stream_buffer_decode) on seeded inputs and the derived bad cases of buffer_cases() and
   records sizes, SHA-256 and return codes in buffer_golden.json.
5. (`make_golden.py trace`) records the reference's lzma_code() return-code sequences
   (LZMA_TELL_* / LZMA_CONCATENATED / LZMA_IGNORE_CHECK flags) for the corpus in stream_trace_golden.json.
6. (`make_golden.py live <reference source tree>`) records what the tests compare with the reference on their own
   inputs (ref_checks_golden.json, ref_xz_*.xz), so that they need neither the reference nor oracle/_ref.
3. Stores the reference's known-answer values for CRC32/CRC64 (tests/test_check.c:74,112) and the
   MicroLZMA encoder KAT (tests/test_microlzma.c:20-32) in kat.json.
"""
import glob, hashlib, json, os, re, shutil, sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import xzlibs as X

REF_FILES = "/root/reference/tests/files"


def buffer_decode_cases():
    """(name, kind, preset, n, mutation) -- tests rebuild the same inputs from the generators.
    mutation: ("trunc", k) drop the last k bytes; ("cap", d) output capacity n + d; ("flags", f);
    ("concat", pad, flags) the Stream twice with `pad` zero bytes between; ("flip", off) xor 0x01 at offset
    (negative = from the end); ("tail", k) k garbage bytes appended; ("nocheck", f) Stream made with
    LZMA_CHECK_NONE, decoded with flags f (LZMA_TELL_NO_CHECK)."""
    cases = []
    for kind, preset, n in (("T", 6, 300000), ("E", 1, 70000), ("R", 3, 65537), ("T", 0, 0), ("T", 3, 1)):
        base = "%s%x_%d" % (kind, preset, n)
        muts = [("cap", 0), ("cap", 5), ("cap", -1), ("trunc", 1), ("trunc", 12), ("trunc", 13), ("trunc", 40), ("tail", 7),
                ("flags", 0x01), ("flags", 0x02), ("flags", 0x04), ("flags", 0x08), ("flags", 0x10), ("flags", 0x20), ("flags", 0x40),
                ("concat", 0, 0x08), ("concat", 8, 0x08), ("concat", 3, 0x08), ("concat", 4, 0x00),
                ("flip", 7), ("flip", 20), ("flip", -3), ("flip", -14), ("nocheck", 0x01), ("nocheck", 0x00), ("nocheck", 0x03)]
        if n > 100:
            muts += [("trunc", 1000), ("cap", -1000), ("flip", 200), ("trunctail", 30000, -1)]
        for m in muts:
            cases.append((base + "_" + "_".join(str(v) for v in m), kind, preset, n, m))
    return cases


def buffer_case_input(kind, preset, n, m, encode):
    """encode(buf, n, preset, check) -> .xz bytes; returns (input bytes, out_cap, flags) of the case."""
    return buffer_apply(encode(X.gendata(kind, n), n, preset, 0 if m[0] == "nocheck" else 4), n, m)


def buffer_apply(xz, n, m):
    """-> (input bytes, out_cap, flags) for one mutation."""
    cap, flags, data = n, 0, xz
    if m[0] == "nocheck":
        flags = m[1]
    if m[0] == "trunc":
        data = xz[: len(xz) - m[1]]
    elif m[0] == "cap":
        cap = max(n + m[1], 0)
    elif m[0] == "flags":
        flags = m[1]
    elif m[0] == "concat":
        data, cap, flags = xz + b"\0" * m[1] + xz, 2 * n, m[2]
    elif m[0] == "flip":
        b = bytearray(xz); b[m[1]] ^= 0x01; data = bytes(b)
    elif m[0] == "tail":
        data = xz + b"\x55" * m[1]
    elif m[0] == "trunctail":  # truncated input AND too small output: whichever the decoder hits first
        data, cap = xz[: len(xz) - m[1]], max(n + m[2], 0)
    return data, cap, flags


def main_buffer():
    assert X.have_ref(), "build oracle/_ref first (make -f oracle/Makefile.ref all)"
    enc = []
    for kind in "TER":
        for preset in (0, 1, 3, 6, 9 | X.XZ_PRESET_EXTREME):
            for n in (0, 1, 5, 4096, 65536, 65537, 300000, 2500000):
                buf = X.gendata(kind, n)
                for check in ((0, 1, 4, 10) if n in (65537, 300000) else (4,)):
                    out = X.ref_buffer_encode(buf, n, preset, check)
                    enc.append({"kind": kind, "preset": preset, "size": n, "check": check, "xz_size": len(out),
                                "xz_sha256": hashlib.sha256(out).hexdigest()})
    enc.append({"kind": "T", "preset": 6, "size": 16 << 20, "check": 4})
    out = X.ref_buffer_encode(X.gendata("T", 16 << 20), 16 << 20, 6, 4)
    enc[-1].update(xz_size=len(out), xz_sha256=hashlib.sha256(out).hexdigest())
    blocks = []
    for kind, preset, n, check in (("T", 6, 0, 4), ("T", 6, 0, 10), ("T", 6, 1, 1), ("T", 6, 300000, 4), ("T", 1, 300000, 10), ("R", 3, 70000, 4),
                                    ("E", 9 | X.XZ_PRESET_EXTREME, 200000, 0), ("T", 6, 65536, 1), ("R", 0, 65537, 10)):
        blk, hs, cs, rc = X.ref_block_buffer_encode(X.gendata(kind, n), n, preset, check)
        blocks.append({"kind": kind, "preset": preset, "size": n, "check": check, "block_size": len(blk), "block_sha256": hashlib.sha256(blk).hexdigest(),
                       "header_size": hs, "compressed_size": cs, "raw_check": rc.hex()})
    dec = {}
    for name, kind, preset, n, m in buffer_decode_cases():
        data, cap, flags = buffer_case_input(kind, preset, n, m, X.ref_buffer_encode)
        r, out, used = X.ref_buffer_decode(data, cap, flags)
        dec[name] = {"ret": r, "in_used": used, "out_size": len(out), "out_sha256": hashlib.sha256(out).hexdigest()}
        print(name, r, used, len(out), flush=True)
    import ctypes as C
    r_ = X.ref(); r_.ref_stream_buffer_bound.restype = C.c_size_t; r_.ref_stream_buffer_bound.argtypes = [C.c_size_t]
    bounds = {str(v): r_.ref_stream_buffer_bound(v) for v in (0, 1, 65536, 65537, 1 << 30, (1 << 63) - 2000, (1 << 63) - 1, (1 << 64) - 1)}
    json.dump({"encode": enc, "decode": dec, "stream_buffer_bound": bounds, "block_buffer_encode": blocks}, open(os.path.join(HERE, "buffer_golden.json"), "w"), indent=1, sort_keys=True)


TRACE_FLAGS = (0x00, 0x01, 0x02, 0x04, 0x08, 0x0C, 0x0B, 0x10, 0x18, 0x20)


def ref_trace(data, flags, cap=1 << 22):
    import ctypes as C
    out = (C.c_uint8 * cap)(); sz = C.c_size_t(); codes = (C.c_uint32 * 32)(); n = C.c_uint32()
    X.ref().ref_decode_trace(data, C.c_size_t(len(data)), C.c_uint32(flags), out, C.c_size_t(cap), C.byref(sz), codes, 32, C.byref(n))
    return [[c & 0xFF, c >> 8] for c in codes[: n.value]], bytes(out[: sz.value])


def main_trace():
    """lzma_stream_decoder + lzma_code(LZMA_FINISH) loop of the reference on every corpus file and a few
    generated multi-Stream inputs, for each flag combination: sequence of (lzma_ret, lzma_get_check)."""
    assert X.have_ref()
    res = {}
    inputs = {n: open(os.path.join(HERE, "ref_files", n), "rb").read() for n in sorted(os.listdir(os.path.join(HERE, "ref_files")))}
    a = X.ref_buffer_encode(X.gendata("T", 50000), 50000, 3, 0)
    b = X.ref_buffer_encode(X.gendata("E", 70000), 70000, 6, 4)
    c = X.ref_encode(X.gendata("R", 40000), 40000, 1, 16384, check=1)
    inputs["gen:none+crc64+crc32mt"] = a + b + c
    inputs["gen:crc64+pad8+none"] = b + bytes(8) + a
    inputs["gen:crc64+pad6+none"] = b + bytes(6) + a
    inputs["gen:none+garbage"] = a + b"garbage!"
    for name, data in inputs.items():
        for fl in TRACE_FLAGS:
            codes, out = ref_trace(data, fl)
            res[f"{name}|{fl:#x}"] = {"codes": codes, "out_size": len(out), "out_sha256": hashlib.sha256(out).hexdigest()}
    json.dump(res, open(os.path.join(HERE, "stream_trace_golden.json"), "w"), indent=0, sort_keys=True)
    print(len(res), "traces")
    # memory limit: LZMA_MEMLIMIT_ERROR, lzma_memusage(), lzma_memlimit_set() too low / exact, then the decode goes on
    import ctypes as C
    mem = {}
    for name in ("good-1-lzma2-1.xz", "good-1-block_header-1.xz", "good-0-empty.xz", "good-2-lzma2.xz", "good-1-check-sha256.xz",
                 "bad-1-lzma2-1.xz", "gen:none+crc64+crc32mt", "gen:crc64+pad8+none"):
        data = inputs[name]
        for fl in (0x00, 0x08, 0x04):
            for ml in (1, 66200 + 4096 - 1, 66200 + (1 << 20), 66200 + (8 << 20) - 1, 66200 + (8 << 20), (1 << 64) - 1):
                out = (C.c_uint8 * (1 << 22))(); sz = C.c_size_t(); codes = (C.c_uint32 * 32)(); n = C.c_uint32(); mu = C.c_uint64()
                X.ref().ref_decode_trace_memlimit(data, C.c_size_t(len(data)), C.c_uint32(fl), C.c_uint64(ml), out, C.c_size_t(1 << 22), C.byref(sz),
                                                  codes, 32, C.byref(n), C.byref(mu))
                mem[f"{name}|{fl:#x}|{ml}"] = {"codes": list(codes[: n.value]), "out_size": sz.value, "memusage": mu.value,
                                               "out_sha256": hashlib.sha256(bytes(out[: sz.value])).hexdigest()}
    json.dump(mem, open(os.path.join(HERE, "memlimit_trace_golden.json"), "w"), indent=0, sort_keys=True)
    print(len(mem), "memlimit traces")


def trace_inputs():
    """Rebuilds the generated inputs of main_trace() from the oracle (bit-identical to the reference)."""
    a = X.oracle_buffer_encode(X.gendata("T", 50000), 50000, 3, 0)
    b = X.oracle_buffer_encode(X.gendata("E", 70000), 70000, 6, 4)
    c = X.oracle_encode(X.gendata("R", 40000), 40000, 1, 16384, check=1)
    return {"gen:none+crc64+crc32mt": a + b + c, "gen:crc64+pad8+none": b + bytes(8) + a, "gen:crc64+pad6+none": b + bytes(6) + a,
            "gen:none+garbage": a + b"garbage!"}


def main_live(ref_tree):
    """What the tests compare with the reference on their own inputs, recorded once so that they run without it:
    ref_checks_golden.json (sizes + SHA-256 of the reference's output, its return codes, struct layouts and symbol
    tables) and two single-threaded `xz -6 -T1` Streams (Blocks without sizes) as ref_xz_*.xz."""
    import ctypes as C
    import random
    import subprocess
    import tempfile
    assert X.have_ref(), "build oracle/_ref first (make -f oracle/Makefile.ref all)"
    sys.path.insert(0, X.ROOT)
    import test_api_cpu as API
    import test_filters_cpu as FC
    import test_gpu_filters as GF
    MiB, KiB = 1 << 20, 1 << 10
    g = {}
    # tests/test_oracle.py
    g["buffer_encode"] = {f"{kind}|{preset:#x}|{n}|{check}": X.digest(X.ref_buffer_encode(X.gendata(kind, n), n, preset, check))
                          for kind, preset, n in (("T", 6, 1234567), ("E", 9 | X.XZ_PRESET_EXTREME, 200001), ("R", 1, 131072), ("L", 3, 700000))
                          for check in (0, 1, 4)}
    g["stream_encode"] = {}
    for kind in "TER":
        for preset, n, bs in ((1, 1 * MiB + 3, 512 * 1024), (6, 600001, 256 * 1024), (3, 700000, 1 * MiB)):
            buf = X.gendata(kind, n)
            xz = X.ref_encode(buf, n, preset, bs)
            r, out = X.ref_decode(xz, n)
            rm, outm = X.ref_decode(xz, n, mt=True)
            g["stream_encode"][f"{kind}|{preset}|{n}|{bs}"] = {"xz": X.digest(xz), "decode": [r] + X.digest(out), "decode_mt": [rm] + X.digest(outm)}
    buf = X.gendata("T", 300000)
    g["match_finders"] = {}
    for mode in (1, 2):
        for mf in (0x03, 0x04, 0x12, 0x13, 0x14):
            for lc, lp, pb in ((3, 0, 2), (0, 2, 0), (4, 0, 4), (1, 3, 1)):
                o = X.LzmaOptions(1 << 20, lc, lp, pb, mode, 32, mf, 0)
                g["match_finders"][f"{mode}|{mf:#x}|{lc}|{lp}|{pb}"] = X.digest(X.ref_encode(buf, 300000, 0, 1 << 20, opts=o))
    xz = X.ref_encode(X.gendata("T", 50000), 50000, 6, 1 << 16)
    bad = bytearray(xz)
    bad[len(xz) // 2] ^= 0x55
    g["truncated"] = {"xz": X.digest(xz), "cut": {str(cut): X.ref_decode(xz[:cut], 50000)[0] for cut in (5, 40, len(xz) // 2, len(xz) - 1)},
                      "flipped": X.ref_decode(bytes(bad), 50000)[0]}
    # tests/test_api_cpu.py
    with tempfile.TemporaryDirectory() as d:
        src, exe = os.path.join(d, "l.c"), os.path.join(d, "l")
        open(src, "w").write(API.LAYOUT_PROG.replace("HEADER", "<lzma.h>"))
        subprocess.check_call(["gcc", "-I", os.path.join(ref_tree, "src", "liblzma", "api"), src, "-o", exe])
        g["lzma_h_layout"] = subprocess.check_output([exe], text=True)
    ref = C.CDLL(os.path.join(X.ROOT, "oracle", "_ref", "liblzma_ref.so"))
    ref.lzma_mt_block_size.restype = C.c_uint64
    g["mt_options"] = {}
    for kw, _ in API.BAD_OPTIONS:
        s = API.LzmaStream()
        g["mt_options"][json.dumps(kw, sort_keys=True)] = ref.lzma_stream_encoder_mt(C.byref(s), C.byref(API._mt(**kw)))
        ref.lzma_end(C.byref(s))
    g["filter_chains"] = {}
    for spec in API.BAD_CHAINS + API.GOOD_CHAINS:
        keep = []
        arr = API._chain(spec, keep)
        s = API.LzmaStream()
        r = ref.lzma_stream_encoder_mt(C.byref(s), C.byref(API._mt(filters=C.cast(arr, C.c_void_p))))
        ref.lzma_end(C.byref(s))
        g["filter_chains"][API.chain_id(spec)] = {"ret": r, "mt_block_size": ref.lzma_mt_block_size(arr) if r == 0 else None}
    # tests/test_filters_cpu.py
    g["bcj"] = {}
    for fid, arg in FC.BCJ_CASES:
        for n in FC.BCJ_SIZES:
            data = FC.codeish(fid, n, 1000 * fid + n)
            g["bcj"][f"{fid}|{arg}|{n}"] = [hashlib.sha256(X.ref_filter_apply(fid, arg, e, data)).hexdigest() for e in (1, 0)]
    g["delta"] = {}
    for dist in FC.DELTA_DISTS:
        for n in FC.DELTA_SIZES:
            rnd = random.Random(dist * 7 + n)
            data = bytes(rnd.getrandbits(8) for _ in range(n))
            g["delta"][f"{dist}|{n}"] = [hashlib.sha256(X.ref_filter_apply(FC.DELTA, dist, e, data)).hexdigest() for e in (1, 0)]
    # tests/test_gpu_filters.py
    data = GF.mixed_input(700 * KiB + 123, 17)
    g["chain_encode"] = {API.chain_id(chain): X.digest(X.ref_chain_encode(data, chain, 6, 256 * KiB)) for chain in GF.CHAINS}
    rnd = random.Random(5)
    data = bytes(rnd.getrandbits(8) for _ in range(300 * KiB))
    g["chain_encode_random"] = {f"{preset}|{API.chain_id(chain)}": X.digest(X.ref_chain_encode(data, chain, preset, 128 * KiB))
                                for preset in (0, 3) for chain in GF.RANDOM_CHAINS}
    # tests/test_gpu_lzma_api.py
    a, b = X.gendata("T", 100000), X.gendata("E", 70000)
    xa, xb = X.ref_encode(a, 100000, 6, 1 << 16), X.ref_encode(b, 70000, 1, 1 << 15)
    g["concat_pad"] = {"inputs": [X.digest(xa), X.digest(xb)]}
    for pad in (0, 8, 6):
        cat = xa + b"\0" * pad + xb
        o2 = (C.c_uint8 * 200000)(); s2 = C.c_size_t()
        g["concat_pad"][str(pad)] = X.ref().ref_decode_flags(cat, C.c_size_t(len(cat)), C.c_uint32(0x08), o2, C.c_size_t(200000), C.byref(s2))
    n = 3 * MiB + 17
    xz = X.ref_buffer_encode(X.gendata("E", n), n, 2, 4)
    r, back, used = X.ref_buffer_decode(xz, n)
    g["buffer_roundtrip"] = {"xz": X.digest(xz), "decode": [r, used] + X.digest(back)}
    xz_cli = os.path.join(X.ROOT, "oracle", "_ref", "xz")
    for name, data in (("T6_300000", bytes(X.gendata("T", 300000)[:300000])), ("zeros_40000000", bytes(40 * 1000 * 1000))):
        st = subprocess.run([xz_cli, "-6", "-T1"], input=data, stdout=subprocess.PIPE, check=True).stdout
        open(os.path.join(HERE, f"ref_xz_{name}_T1.xz"), "wb").write(st)
    # tests/test_hybrid_cpu.py: the lzma_* symbols the reference `xz` imports and the ones the reference liblzma defines
    def syms(path, flag):
        out = subprocess.run(["nm", "-D", flag, path], stdout=subprocess.PIPE, text=True, check=True).stdout
        return sorted({ln.split()[-1] for ln in out.splitlines() if re.search(r"\blzma_", ln)})
    g["xz_imports"] = syms(xz_cli, "--undefined-only")
    g["ref_liblzma_exports"] = syms(os.path.join(X.ROOT, "oracle", "_ref", "liblzma_ref.so"), "--defined-only")
    json.dump(g, open(os.path.join(HERE, "ref_checks_golden.json"), "w"), indent=0, sort_keys=True)


def main():
    assert X.have_ref(), "build oracle/_ref first (make -f oracle/Makefile.ref all)"
    dst = os.path.join(HERE, "ref_files")
    os.makedirs(dst, exist_ok=True)
    verdicts = {}
    for f in sorted(glob.glob(os.path.join(REF_FILES, "*.xz"))):
        name = os.path.basename(f)
        data = open(f, "rb").read()
        if len(data) > 64 * 1024:
            continue  # good-1-delta-lzma2.tiff.xz: big and a Delta chain (out of scope)
        shutil.copyfile(f, os.path.join(dst, name))
        r, out = X.ref_decode(data, 1 << 22)
        verdicts[name] = {"ret": r, "out_size": len(out), "out_sha256": hashlib.sha256(out).hexdigest() if r == 0 else None}
        # same with LZMA_CONCATENATED (what `xz -d` uses): Stream Padding / multi-Stream verdicts
        import ctypes as C
        o2 = (C.c_uint8 * (1 << 22))(); s2 = C.c_size_t()
        r2 = X.ref().ref_decode_flags(data, C.c_size_t(len(data)), C.c_uint32(0x08), o2, C.c_size_t(1 << 22), C.byref(s2))
        verdicts[name]["ret_concat"] = r2
        verdicts[name]["out_concat_sha256"] = hashlib.sha256(bytes(o2[: s2.value])).hexdigest() if r2 == 0 else None
    json.dump(verdicts, open(os.path.join(HERE, "decode_verdicts.json"), "w"), indent=1, sort_keys=True)

    enc = []
    MiB = 1 << 20
    cases = []
    for kind in "TER":
        for preset in (0, 1, 3, 4, 6, 9 | X.XZ_PRESET_EXTREME):
            for n in (0, 1, 2, 3, 4, 5, 273, 4096, 65535, 65536, 65537, 300000):
                cases.append((kind, preset, n, 256 * 1024))
        for preset in (1, 3, 6):
            cases.append((kind, preset, 2 * MiB - 273, 4 * MiB))
            cases.append((kind, preset, 2 * MiB + 273, 1 * MiB))
            cases.append((kind, preset, 3 * MiB + 1, MiB))
    # BASELINE.json configs[0] exactly, plus one full 16 MiB block per GPU config's preset
    cases += [("T", 1, 16 * MiB, 16 * MiB), ("T", 6, 16 * MiB, 16 * MiB), ("T", 6, 16 * MiB + 1, 16 * MiB),
              ("R", 3, 16 * MiB, 16 * MiB), ("E", 6, 16 * MiB, 16 * MiB), ("E", 9 | X.XZ_PRESET_EXTREME, 4 * MiB, 16 * MiB)]
    for kind, preset, n, bs in cases:
        buf = X.gendata(kind, n)
        out = X.ref_encode(buf, n, preset, bs)
        enc.append({"kind": kind, "preset": preset, "size": n, "block_size": bs, "check": 4,
                    "xz_size": len(out), "xz_sha256": hashlib.sha256(out).hexdigest()})
        print(kind, hex(preset), n, bs, len(out), flush=True)
    json.dump(enc, open(os.path.join(HERE, "encode_golden.json"), "w"), indent=1)

    kat = {"crc32_123456789": 0xCBF43926, "crc64_123456789": 0x995DC9BBDF1939FA,
           "ref_crc32_123456789": X.ref().ref_crc32(b"123456789", 9, 0),
           "ref_crc64_123456789": X.ref().ref_crc64(b"123456789", 9, 0),
           "microlzma_hello_world_crc32": 0x3CDE40A8}
    json.dump(kat, open(os.path.join(HERE, "kat.json"), "w"), indent=1)


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "buffer":
        main_buffer()
    elif len(sys.argv) > 1 and sys.argv[1] == "trace":
        main_trace()
    elif len(sys.argv) > 2 and sys.argv[1] == "live":
        main_live(sys.argv[2])
    else:
        main()
