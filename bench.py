#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on BASELINE.json's config.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--config 1|4|5] [--dump-outputs DIR]

Workloads (config.workload names the one that ran):
  --config 1 (default): configs[1] = "xz -6 bt4, 8 MiB dict, 1 GiB synthetic text, 64 .xz blocks" (16 MiB
      blocks, CRC64) on ONE GPU.  At N GPUs the job is WEAK-scaled (per-GPU work fixed): an N GiB text of
      64*N Blocks, rank r owns Blocks [64r, 64r+64) -- the Blocks-per-GPU of BASELINE's own 8-GPU configs
      (configs[3]: 32, configs[4]: 64).  `--scaling strong` keeps the job at 1 GiB (rank r owns Blocks
      [r*64/N, (r+1)*64/N)); that job is latency-flat in N by construction (one Block = one serial chain,
      one GPU already runs all 64 side by side; measured: profiles/bench_r02_2gpu.json).  The decode legs
      are configs[2] (the Stream this run just produced).
  --config 4: configs[3] = "-9e bt4, 4 GiB enwik-style, 256 blocks", fixed job sharded over N GPUs (strong).
  --config 5: configs[4] = "-3 hc4, 8 GiB incompressible, 512 blocks", fixed job sharded over N GPUs (strong).
The only exchange between ranks is one all-gather of the 16-byte Index records (NCCL).

A step = ONE encode pass of the hot path over this rank's Blocks through the reference-facing
host-buffer call (xzb_encode_blocks_host: pinned host input -> finished Blocks + Index records in
host memory; the worker_encode() cut of stream_encoder_mt.c:218-359):
  * `e2e.value` : MB/s (1e6 B of input / s), wall clock around the call + the record gather, barriers
                  and device synchronisation on both sides, host<->device copies inside; max over ranks;
  * `value`     : the same pass timed ON THE DEVICE by the library's own CUDA events with the input
                  already in HBM (ms_total - ms_h2d - ms_d2h of that call), max over ranks;
  * `e2e_lzma_code` (N = 1): one extra pass through lzma_stream_encoder_mt + lzma_code(LZMA_FINISH) of
                  the liblzma-named shim -- the call the reference arm makes -- wall clock;
  * `decode`    : decode MB/s of the Stream just produced, device-timed and e2e;
  * `roofline`  : the match-finder kernel (CUDA events on the stream it runs on);
  * `parity`    : SHA-256 of EVERY Block against tests/golden/bench_golden.json (recorded from the
                  unmodified reference), plus decode(encode(x)) == x;
  * `cpu_baseline` (N = 1, rank 0): the unmodified reference (oracle/_ref, lzma_stream_encoder_mt,
                  all host threads) on a bounded sample of the same Blocks; its output is checked
                  against the same golden vectors.
`--impl reference` times the UNMODIFIED reference on a bounded sample per step and says which.
Inputs (>= 128 MiB per GPU) exceed the 126 MB L2 => no explicit L2 flush between timed iterations.
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

MiB = 1 << 20
XZ_EXTREME = 0x80000000
CONFIGS = {
    # id: (metric text, kind, preset, total bytes, golden name)
    1: ("encode MB/s at -6, 1 GiB synthetic text per GPU, 64 x 16 MiB .xz blocks (bit-exact); decode MB/s beside it", "T", 6, 1024 * MiB, "T6"),
    4: ("encode MB/s at -9e, 4 GiB enwik-style synthetic, 256 x 16 MiB .xz blocks (bit-exact)", "E", 9 | XZ_EXTREME, 4096 * MiB, "E9e"),
    5: ("encode MB/s at -3, 8 GiB incompressible synthetic, 512 x 16 MiB .xz blocks (bit-exact)", "R", 3, 8192 * MiB, "R3"),
}


def measured_hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(is_bt, kind, n_positions):
    """dram__bytes_read.sum + dram__bytes_write.sum of the match-finder kernel, per step, from the
    `ncu --set full` capture named in profiles/ncu_traffic.json (bytes per inserted position of that
    capture x the positions of this step).  None when no capture exists for the workload."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.exists(p):
        return None, None
    try:
        db = json.load(open(p))
        e = db.get(("bt_" if is_bt else "hc_") + kind)
        if not e:
            return None, None
        return float(e["dram_bytes_per_position"]) * n_positions, e.get("capture")
    except Exception:
        return None, None


def load_golden(name):
    p = os.path.join(ROOT, "tests", "golden", "bench_golden.json")
    if not os.path.exists(p):
        return None
    return json.load(open(p)).get(name)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for i, nme in enumerate(names):
                if f[2 + i].lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def host_threads_info():
    """Threads the host really offers this process (affinity mask, cgroup CPU quota)."""
    info = {"os_cpu_count": os.cpu_count()}
    try:
        info["affinity"] = len(os.sched_getaffinity(0))
    except Exception:
        pass
    for p in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            info["cgroup_" + os.path.basename(p)] = open(p).read().strip()
            break
        except Exception:
            pass
    return info


def workload_config(args, note=None):
    kinds = {'T': 'Lorem-word text, tests/create_compress_files.c generator scaled', 'E': 'enwik-style', 'R': 'random'}
    c = {"workload": f"xz -{args.preset & 0x1F}{'e' if args.preset & XZ_EXTREME else ''} LZMA2, {args.size // MiB} MiB synthetic '{args.kind}' "
                     f"({kinds[args.kind]}), {args.size // args.block_size} x {args.block_size // MiB} MiB .xz blocks, CRC64",
         "baseline_config": args.config, "preset": args.preset & 0x1F, "extreme": bool(args.preset & XZ_EXTREME),
         "block_size": args.block_size, "total_bytes": args.size, "check": "crc64",
         "l2_policy": "inputs (>= 128 MiB per GPU) exceed the 126 MB L2; no explicit flush"}
    if args.scaling == "weak" and args.world > 1:
        c["workload"] += f" = {args.world} GPUs x {args.size // args.world // MiB} MiB ({args.size // args.block_size // args.world} Blocks per GPU, weak scaling)"
    if note:
        c["workload"] += "; " + note
        c["sample"] = note
    return c


def block_hashes(buf, recs):
    """[(total_size, sha256)] of consecutive Blocks in `buf` given their Index records (unpadded sizes)."""
    out, pos = [], 0
    for unpadded, _ in recs:
        total = (unpadded + 3) // 4 * 4
        out.append([total, hashlib.sha256(buf[pos:pos + total]).hexdigest()])
        pos += total
    return out


DUMP_SAMPLE = 8 * MiB  # encoded bytes kept by --dump-outputs (32 MB as float32)


def dump_outputs(out_dir, blocks, recs):
    """What the timed encode returned in its last step, as arrays two builds can be compared with:
    index_records.npy  (unpadded size, uncompressed size) of every Block, float64 (exact below 2**53);
    block_sha256.npy   SHA-256 of every Block, one row of 32 bytes per Block, float32;
    blocks_sample.npy  the encoded bytes at DUMP_SAMPLE positions drawn with a fixed seed (all bytes when
                       there are fewer), float32."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "index_records.npy"), np.array(recs, dtype=np.float64).reshape(-1, 2))
    sha = [np.frombuffer(bytes.fromhex(h), dtype=np.uint8) for _, h in block_hashes(blocks.tobytes(), recs)]
    np.save(os.path.join(out_dir, "block_sha256.npy"), np.array(sha, dtype=np.float32).reshape(-1, 32))
    if len(blocks) > DUMP_SAMPLE:
        blocks = blocks[np.sort(np.random.default_rng(0).integers(0, len(blocks), DUMP_SAMPLE))]
    np.save(os.path.join(out_dir, "blocks_sample.npy"), blocks.astype(np.float32))


def run_reference(args):
    """Reference arm: lzma_stream_encoder_mt of the unmodified reference on the host cores."""
    import xzlibs as X
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if not X.have_ref():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libref_shim.so is not built"}))
        return
    cores = X.ref().ref_cputhreads() or os.cpu_count() or 1
    nblocks_total = args.size // args.block_size
    # One step = one pass of lzma_stream_encoder_mt (all host threads) over the first `sample_blocks`
    # Blocks of the workload.  The whole 64-Block workload takes about a minute per pass on the GPU
    # box's host, so with the driver's 25 passes the sample is bounded to keep the run within minutes.
    passes = args.warmup + args.steps
    sample_blocks = args.ref_blocks if args.ref_blocks else (nblocks_total if passes <= 3 else 16)
    sample_blocks = max(1, min(nblocks_total, sample_blocks))
    n = sample_blocks * args.block_size
    buf = X.gendata(args.kind, n)
    times = []
    out = b""
    for it in range(passes):
        t = time.perf_counter()
        out = X.ref_encode(buf, n, args.preset, args.block_size, threads=0)
        dt = time.perf_counter() - t
        if it >= args.warmup:
            times.append(dt)
    t_step = sum(times) / len(times)
    val = n / 1e6 / t_step
    dbuf = (C.c_uint8 * n)(); dsz = C.c_size_t()
    t = time.perf_counter()
    r = X.ref().ref_decode_mt(out, C.c_size_t(len(out)), C.c_uint32(0), dbuf, C.c_size_t(n), C.byref(dsz))
    dt_dec = time.perf_counter() - t
    sample = (f"reference arm timed on the first {sample_blocks} of the {nblocks_total} Blocks ({n // MiB} MiB) per step, "
              f"lzma_stream_encoder_mt threads={cores}, buffers in RAM")
    line = {
        "impl": "reference", "metric": args.metric, "value": val, "unit": "MB/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": t_step * 1e3, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": workload_config(args, sample),
        "cpu_baseline": {"value": val, "unit": "MB/s", "cores": int(cores), "kind": "reference", "sample": sample,
                         "host": host_threads_info()},
        "e2e": {"value": val, "unit": "MB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "decode": {"value": n / 1e6 / dt_dec if r == 0 else None, "unit": "MB/s", "note": "lzma_stream_decoder_mt, same sample"},
        "xz_bytes": len(out),
    }
    print(json.dumps(line))


def lzma_code_pass(h_in_ptr, n, preset, bs, h_out_ptr, cap):
    """One pass through the liblzma-named entry points of libxzb200.so, as src/xz/coder.c drives them:
    lzma_stream_encoder_mt(&strm, &mt); lzma_code(&strm, LZMA_FINISH) until LZMA_STREAM_END; lzma_end."""
    import xz_b200
    from xz_b200 import liblzma as LZ
    return LZ.encode_mt(h_in_ptr, n, preset, bs, h_out_ptr, cap)


def _device(local_rank):
    import torch
    return torch.device("cuda", local_rank)


def _init_group(local_rank):
    import torch.distributed as dist
    dist.init_process_group("nccl", device_id=_device(local_rank))


def run_ours(args):
    import torch
    import torch.distributed as dist
    import __graft_entry__ as ge
    import xz_b200
    from xz_b200 import sharding
    import xzlibs as X

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if rank == 0:
        ge.build()
    if world > 1:
        torch.cuda.set_device(local_rank)
        # NCCL announces its version on stdout when the first communicator is made; stdout carries ONE JSON line, so the
        # file descriptor points at stderr while the group comes up
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            _init_group(local_rank)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)
    if rank != 0:
        ge.build()
    torch.cuda.set_device(local_rank)
    ctx = xz_b200.Context(local_rank)
    opts = xz_b200.lzma_lzma_preset(args.preset)
    bs = args.block_size
    nblocks = args.size // bs
    lo, hi = sharding.shard_blocks(nblocks, world, rank)
    my_blocks = hi - lo
    my_off = lo * bs
    my_n = my_blocks * bs

    # synthetic shard, generated on the host (excluded from all timings), pinned
    h_in = torch.empty(my_n, dtype=torch.uint8).pin_memory()
    assert X.gen().xzgen_fill(C.c_char(args.kind.encode()), C.c_void_p(h_in.data_ptr()), C.c_size_t(my_n), C.c_uint64(my_off)) == 0
    cap = my_blocks * xz_b200.lzma_block_buffer_bound(bs) + 4096
    h_out = torch.empty(cap, dtype=torch.uint8).pin_memory()
    dev = _device(local_rank)
    torch.cuda.synchronize()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce(x, op):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=op)
        return float(t.item())

    def rmax(x):
        return reduce(x, dist.ReduceOp.MAX) if world > 1 else x

    def rsum(x):
        return reduce(x, dist.ReduceOp.SUM) if world > 1 else x

    dev_times, e2e_times = [], []
    stat_acc = {}
    launches = 0
    sampler = ClockSampler(local_rank)
    all_recs, recs, size_h = None, None, 0
    total_steps = args.warmup + args.steps
    for it in range(total_steps):
        timed = it >= args.warmup
        if it == args.warmup and rank == 0:
            sampler.start()
        barrier()
        t0 = time.perf_counter()
        size_h, recs = ctx.encode_blocks_host(h_in.data_ptr(), my_n, opts, 4, bs, h_out.data_ptr(), cap)
        all_recs = sharding.gather_records(recs, device=dev)  # the one exchange step of the path
        barrier()
        t1 = time.perf_counter()
        if timed:
            s = ctx.stats().as_dict()
            e2e_times.append(t1 - t0)
            dev_times.append((s["ms_total"] - s["ms_h2d"] - s["ms_d2h"]) / 1e3)
            launches += s["gpu_launches"]
            for k, v in s.items():
                stat_acc[k] = stat_acc.get(k, 0) + v
    clocks = sampler.stop() if rank == 0 else None
    n_steps = len(dev_times)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, h_out[:size_h].numpy(), recs)

    # ---- parity: every Block of this rank against the reference's golden vectors ----
    mine = h_out[:size_h].numpy().tobytes()
    got = block_hashes(mine, recs)
    gold = load_golden(args.golden) if args.golden else None
    checked = bad = 0
    if gold and gold["block_size"] == bs and gold["preset"] == args.preset and gold["kind"] == args.kind:
        for i, g in enumerate(got):
            if lo + i < gold["nblocks"]:
                checked += 1
                bad += g != gold["blocks"][lo + i]
    checked_all, bad_all = int(rsum(checked)), int(rsum(bad))

    # ---- decode legs on this rank's shard (configs[2]); also the round-trip property for every Block ----
    idx = xz_b200.index_encode(recs)
    stream = xz_b200.stream_header(4) + mine + idx + xz_b200.stream_footer(4, len(idx))
    h_xz = torch.frombuffer(bytearray(stream), dtype=torch.uint8).pin_memory()
    h_back = torch.empty(my_n, dtype=torch.uint8).pin_memory()
    dec_e2e, dec_dev = [], []
    for it in range(3):
        barrier()
        t0 = time.perf_counter()
        r, sz = ctx.stream_decode_into(h_xz.data_ptr(), len(stream), h_back.data_ptr(), my_n)
        barrier()
        t1 = time.perf_counter()
        assert r == 0 and sz == my_n
        if it > 0:
            dec_e2e.append(t1 - t0)
            sd = ctx.stats().as_dict()
            dec_dev.append((sd["ms_total"] - sd["ms_h2d"] - sd["ms_d2h"]) / 1e3)
    roundtrip_ok = bool(torch.equal(h_back, h_in))
    roundtrip_all = int(rsum(0 if roundtrip_ok else 1)) == 0

    # ---- N = 1: one pass through lzma_stream_encoder_mt + lzma_code (the reference arm's own call) ----
    lzma_code = None
    if world == 1 and not args.no_lzma_code:
        ctx.close()  # the shim owns its own context (worker pool); free this one's HBM workspace first
        os.environ["XZB_DEVICE"] = str(local_rank)  # this line measures ONE GPU (the shim would otherwise fan out over all visible ones)
        try:
            t0 = time.perf_counter()
            out_len = lzma_code_pass(h_in.data_ptr(), my_n, args.preset, bs, h_out.data_ptr(), cap)
            dt = time.perf_counter() - t0
            same = h_out[:out_len].numpy().tobytes() == stream
            lzma_code = {"value": my_n / 1e6 / dt, "unit": "MB/s", "ms": dt * 1e3, "stream_identical": bool(same),
                         "note": "lzma_stream_encoder_mt + lzma_code(LZMA_FINISH) on host buffers, one pass, wall clock"}
        except Exception as ex:  # the number is optional, the failure is not hidden
            lzma_code = {"error": repr(ex)}

    t_dev = rmax(sum(dev_times) / n_steps)
    t_e2e = rmax(sum(e2e_times) / n_steps)
    t_dec_dev = rmax(sum(dec_dev) / len(dec_dev))
    t_dec_e2e = rmax(sum(dec_e2e) / len(dec_e2e))
    total_launches = rsum(launches)
    xz_total = rsum(size_h)
    ms_mf = stat_acc.get("ms_mf", 0) / n_steps
    ms_parse = stat_acc.get("ms_parse", 0) / n_steps
    ms_prep = stat_acc.get("ms_mf_prep", 0) / n_steps
    mf_bytes = stat_acc.get("mf_bytes_algorithmic", 0) / n_steps
    is_bt = bool(opts.mf & 0x10)
    peak, peak_src = measured_hbm_peak()
    mf_gbs = mf_bytes / 1e9 / (ms_mf / 1e3) if ms_mf > 0 else 0.0
    traffic, traffic_src = ncu_traffic(is_bt, args.kind, mf_bytes / (33.0 if is_bt else 29.0))

    if rank == 0:
        cpu_baseline = None
        if world == 1 and not args.no_cpu_baseline and X.have_ref():
            cores = X.ref().ref_cputhreads()
            sample_blocks = max(1, min(my_blocks, args.cpu_blocks))
            n_s = sample_blocks * bs
            sbuf = h_in.numpy().ctypes.data_as(C.POINTER(C.c_uint8))
            t0 = time.perf_counter()
            ref_xz = X.ref_encode(sbuf, n_s, args.preset, bs, threads=0)
            dt = time.perf_counter() - t0
            # the reference's output for these Blocks is exactly what the GPU produced
            ref_blocks_len = sum(t for t, _ in got[:sample_blocks])
            ref_same = ref_xz[12:12 + ref_blocks_len] == mine[:ref_blocks_len]
            dbuf = (C.c_uint8 * my_n)(); dsz = C.c_size_t()
            t0 = time.perf_counter()
            rr = X.ref().ref_decode_mt(stream, C.c_size_t(len(stream)), C.c_uint32(0), dbuf, C.c_size_t(my_n), C.byref(dsz))
            dt_dec = time.perf_counter() - t0
            dec_ref = my_n / 1e6 / dt_dec if rr == 0 and dsz.value == my_n else None
            del dbuf
            cpu_baseline = {"value": n_s / 1e6 / dt, "decode_value": dec_ref, "unit": "MB/s", "cores": int(cores), "kind": "reference",
                            "sample": f"first {sample_blocks} of the {nblocks} Blocks ({n_s // MiB} MiB), one pass, lzma_stream_encoder_mt "
                                      f"(oracle/_ref) threads={cores}; decode_value: lzma_stream_decoder_mt over the whole Stream",
                            "output_identical_to_gpu": bool(ref_same), "host": host_threads_info()}
        if checked_all:
            parity = f"bit-exact ({checked_all - bad_all}/{checked_all} Blocks vs reference golden SHA-256)" if bad_all == 0 \
                else f"MISMATCH ({bad_all} of {checked_all} Blocks differ from the reference)"
            if checked_all < nblocks:
                parity += f" [the golden file holds the first {checked_all} of this job's {nblocks} Blocks; the rest: round trip only]"
        else:
            parity = "no golden vector for this workload"
        parity += "; decode(encode(x)) == x for every Block" if roundtrip_all else "; ROUND TRIP FAILED"
        line = {
            "metric": args.metric, "value": args.size / 1e6 / t_dev, "unit": "MB/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": t_dev * 1e3, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": workload_config(args),
            "e2e": {"value": args.size / 1e6 / t_e2e, "unit": "MB/s", "h2d_bytes_per_step": args.size, "d2h_bytes_per_step": int(xz_total),
                    "ms_per_step": t_e2e * 1e3, "api": "xzb_encode_blocks_host (worker_encode cut) + Index record all-gather"},
            "e2e_lzma_code": lzma_code,
            "decode": {"value": args.size / 1e6 / t_dec_dev, "e2e_value": args.size / 1e6 / t_dec_e2e, "unit": "MB/s",
                       "h2d_bytes_per_step": int(xz_total), "d2h_bytes_per_step": args.size},
            "gpu_launches": int(total_launches),
            "roofline": {"kernel": "xzb_k_bt (match finder)" if is_bt else "xzb_k_hc (match finder)", "bound": "hbm",
                         "achieved": mf_gbs, "peak": peak, "unit": "GB/s", "frac": mf_gbs / peak if peak else None,
                         "traffic": traffic, "traffic_source": traffic_src,
                         "peak_source": peak_src, "bytes_per_launch": mf_bytes, "ms_per_launch": ms_mf,
                         "note": "algorithmic bytes = inserted positions x (29 hc | 33 bt) B (SURVEY 8d lower bound); rank 0's shard; "
                                 "time = CUDA events on the stream the match finder runs on, summed over the step's launches"},
            "kernels_ms": {"mf_prep(sort+heads)": ms_prep, "match_finder": ms_mf, "parse+rangecode": ms_parse,
                           "other": stat_acc.get("ms_other", 0) / n_steps},
            "cpu_baseline": cpu_baseline,
            "clocks": clocks,
            "parity": parity,
            "xz_bytes": int(xz_total) + 12 + len(xz_b200.index_encode(all_recs)) + 12,
            "index_records": len(all_recs),
        }
        if args.config == 1 and args.scaling == "weak":
            line["scaling_note"] = ("weak: 64 Blocks (1 GiB) per GPU at every N, no data-path collective.  The fixed 64-Block job (--scaling strong) is "
                                    "latency-flat in N: one Block = one serial chain and one GPU already runs all 64 side by side "
                                    "(N=2 measured 89.9 MB/s vs 88.9 at N=1, profiles/bench_r02_2gpu.json)")
        elif nblocks // world <= 64 and is_bt:
            line["scaling_note"] = ("64 Blocks = 64 serial chains: one GPU already runs them all side by side, so the step time is one "
                                    "Block's parse at any N (latency-flat by construction)")
        print(json.dumps(line))
    ctx.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=1, choices=sorted(CONFIGS))
    ap.add_argument("--size", type=int, default=0, help="total bytes (default: the config's)")
    ap.add_argument("--block-size", type=int, default=16 * MiB)
    ap.add_argument("--preset", type=lambda s: int(s, 0), default=None)
    ap.add_argument("--kind", default=None)
    ap.add_argument("--cpu-blocks", type=int, default=16, help="Blocks of the in-run reference pass (cpu_baseline)")
    ap.add_argument("--ref-blocks", type=int, default=0, help="--impl reference: Blocks per step (0 = automatic bound)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-lzma-code", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write rank 0's output of the last timed step to DIR/*.npy (records, per-Block SHA-256, seeded byte sample)")
    ap.add_argument("--scaling", default=None, choices=["weak", "strong"],
                    help="N > 1: weak = the config's job per GPU (default for --config 1), strong = the config's job split over the GPUs")
    args = ap.parse_args()
    metric, kind, preset, size, golden = CONFIGS[args.config]
    args.metric = metric
    args.golden = golden if (args.kind in (None, kind) and args.preset in (None, preset)) else None
    args.kind = args.kind or kind
    args.preset = preset if args.preset is None else args.preset
    args.size = args.size or size
    args.world = int(os.environ.get("WORLD_SIZE", "1"))
    args.scaling = args.scaling or ("weak" if args.config == 1 else "strong")
    if args.scaling == "weak":
        args.size *= args.world  # rank r owns the r-th `size` bytes of the N x size job
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
