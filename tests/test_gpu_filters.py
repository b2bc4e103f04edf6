"""Delta / BCJ filter chains on the GPU path (-m gpu): Streams made with chains are byte-identical to the unmodified
reference's lzma_stream_encoder_mt with the same chain on the same inputs (size and SHA-256 recorded in
tests/golden/ref_checks_golden.json), and those Streams decode to the input through xzb_k_decode + xzb_k_filter."""
import random

import pytest

import xzlibs as X
from test_api_cpu import chain_id

pytestmark = pytest.mark.gpu
DELTA, X86, POWERPC, IA64, ARM, ARMTHUMB, SPARC, ARM64, RISCV = 3, 4, 5, 6, 7, 8, 9, 10, 11
KiB = 1 << 10


@pytest.fixture(scope="module")
def ctx():
    import xz_b200
    c = xz_b200.Context(0)
    yield c
    c.close()


def mixed_input(n, seed):
    """Text, a ramp (delta-friendly), and random bytes salted with branch opcodes of every architecture."""
    from test_filters_cpu import codeish
    rnd = random.Random(seed)
    parts = []
    t = bytes(X.gendata("T", n // 3)[: n // 3])
    parts.append(t)
    parts.append(bytes((i * 3 + (i >> 8)) & 0xFF for i in range(n // 3)))
    rest = n - 2 * (n // 3)
    per = rest // 9
    for fid in (X86, ARM, ARMTHUMB, POWERPC, SPARC, ARM64, IA64, RISCV):
        parts.append(codeish(fid, per, seed + fid))
    parts.append(bytes(rnd.getrandbits(8) for _ in range(rest - 8 * per)))
    return b"".join(parts)


CHAINS = [[(DELTA, 1)], [(DELTA, 4)], [(DELTA, 256)], [(X86, 0)], [(X86, 0x1000)], [(ARM, 0)], [(ARMTHUMB, 0)], [(POWERPC, 0)], [(SPARC, 0)],
          [(ARM64, 0)], [(ARM64, 0x40000)], [(IA64, 0)], [(RISCV, 0)], [(RISCV, 0x2000), (DELTA, 2)], [(DELTA, 2), (X86, 0)], [(ARM64, 0), (DELTA, 4)], [(X86, 0), (DELTA, 1), (ARM, 0)]]
RANDOM_CHAINS = [[(X86, 0)], [(DELTA, 3), (ARM64, 0)]]


@pytest.mark.parametrize("chain", CHAINS, ids=chain_id)
def test_chain_encode_identical_and_decode(ctx, chain):
    n = 700 * KiB + 123
    data = mixed_input(n, 17)
    ctx.set_filters(chain)
    try:
        got = ctx.stream_encode(data, preset=6, block_size=256 * KiB, n=n)
    finally:
        ctx.set_filters(())
    assert X.digest(got) == X.ref_golden()["chain_encode"][chain_id(chain)]
    r, back = ctx.stream_decode(got, n)
    assert r == 0 and back == data


@pytest.mark.parametrize("preset", [0, 3])
def test_chain_fast_presets_and_incompressible_fallback(ctx, preset):
    """Random bytes: every Block falls back to uncompressed LZMA2 chunks of the UNFILTERED input under an LZMA2-only
    header (block_buffer_encoder.c:87-162), whatever the chain says."""
    n = 300 * KiB
    rnd = random.Random(5)
    data = bytes(rnd.getrandbits(8) for _ in range(n))
    for chain in RANDOM_CHAINS:
        ctx.set_filters(chain)
        try:
            got = ctx.stream_encode(data, preset=preset, block_size=128 * KiB, n=n)
        finally:
            ctx.set_filters(())
        assert X.digest(got) == X.ref_golden()["chain_encode_random"][f"{preset}|{chain_id(chain)}"]
        r, back = ctx.stream_decode(got, n)
        assert r == 0 and back == data


def test_bad_chains_are_refused(ctx):
    import xz_b200
    for chain in ([(DELTA, 0)], [(DELTA, 257)], [(ARM, 2)], [(IA64, 8)], [(RISCV, 1)], [(0x0C, 0)], [(0x21, 0)], [(X86, 0)] * 4):
        with pytest.raises(xz_b200.XzError):
            ctx.set_filters(chain)
    ctx.set_filters(())
