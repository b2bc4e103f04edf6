"""CPU dry run of bench.py's host glue (argument handling, Block sharding, the Index record gather, the
JSON line) for tests/test_bench_glue_cpu.py: torch.cuda and the GPU context are replaced by stand-ins --
the stand-in context encodes with the oracle (oracle/liboracle.so, the CPU restatement of the reference), so the
run needs no GPU and says nothing about the product path.  Launched under torch.distributed.run with the gloo backend."""
import ctypes as C
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import torch
import torch.distributed as dist

import bench
import xz_b200
import xzlibs as X

def _vli(b, pos):
    v = shift = 0
    while True:
        c = b[pos]; pos += 1
        v |= (c & 0x7F) << shift; shift += 7
        if not c & 0x80:
            return v, pos


class FakeContext:
    """Same method names and return shapes as xz_b200.Context; Blocks come from the oracle on the CPU."""

    def __init__(self, device=0):
        self._stats = {}

    def close(self):
        pass

    def stats(self):
        st = self._stats

        class S:
            def as_dict(self_inner):
                return dict(st)
        return S()

    def encode_blocks_host(self, src, n, opts, check, block_size, dst, cap):
        t0 = time.perf_counter()
        data = C.string_at(src, n)
        out, recs = b"", []
        for off in range(0, n, block_size):
            blk = data[off:off + block_size]
            buf = (C.c_uint8 * len(blk)).from_buffer_copy(blk)
            xz = X.oracle_encode(buf, len(blk), 0, block_size, opts=opts)
            index_size = (int.from_bytes(xz[-8:-4], "little") + 1) * 4
            body = xz[12:len(xz) - 12 - index_size]
            idx = xz[len(xz) - 12 - index_size:]
            cnt, p = _vli(idx, 1)
            assert cnt == 1
            unpadded, p = _vli(idx, p)
            uncomp, p = _vli(idx, p)
            assert uncomp == len(blk) and (unpadded + 3) // 4 * 4 == len(body)
            out += body
            recs.append((unpadded, uncomp))
        assert len(out) <= cap
        C.memmove(dst, out, len(out))
        ms = (time.perf_counter() - t0) * 1e3
        self._stats = {"ms_total": ms, "ms_h2d": 0.0, "ms_d2h": 0.0, "ms_mf_prep": 0.0, "ms_mf": ms / 2, "ms_parse": ms / 2, "ms_other": 0.0,
                       "gpu_launches": 0, "mf_bytes_algorithmic": 33 * n}
        return len(out), recs

    def stream_decode_into(self, src, n, dst, cap):
        t0 = time.perf_counter()
        r, out = X.oracle_decode(C.string_at(src, n), cap)
        C.memmove(dst, out, len(out))
        ms = (time.perf_counter() - t0) * 1e3
        self._stats = {"ms_total": ms, "ms_h2d": 0.0, "ms_d2h": 0.0}
        return r, len(out)


def main():
    torch.cuda.set_device = lambda *a, **k: None
    torch.cuda.synchronize = lambda *a, **k: None
    torch.Tensor.pin_memory = lambda self, *a, **k: self
    bench._device = lambda local_rank: torch.device("cpu")
    bench._init_group = lambda local_rank: dist.init_process_group("gloo")
    xz_b200.Context = FakeContext
    bench.main()


if __name__ == "__main__":
    main()
