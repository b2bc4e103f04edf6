"""bench.py's host glue at world sizes 1 and 2 without a GPU (tests/bench_glue_harness.py puts an oracle-backed
stand-in where the GPU context is): the sharding of the job, the record gather, the printed JSON line.  The numbers
it prints are the oracle's on the CPU and mean nothing; the shape of the line and the job arithmetic are the test."""
import json
import os
import socket
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HARNESS = os.path.join(ROOT, "tests", "bench_glue_harness.py")
MiB = 1 << 20


def _port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close()
    return p


def _run(world, extra):
    common = ["--gpus", str(world), "--steps", "1", "--warmup", "1", "--size", str(4 * MiB), "--block-size", str(MiB), "--preset", "0",
              "--no-cpu-baseline", "--no-lzma-code"] + extra
    if world == 1:
        cmd = [sys.executable, HARNESS] + common
    else:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
               "--master-port", str(_port()), HARNESS] + common
    env = dict(os.environ)
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"):
        env.pop(k, None)
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, r.stdout   # ONE JSON line, from rank 0
    return json.loads(lines[0])


def test_one_gpu_line():
    ln = _run(1, [])
    assert ln["n_gpus"] == 1 and ln["config"]["total_bytes"] == 4 * MiB and ln["index_records"] == 4
    assert ln["e2e"]["h2d_bytes_per_step"] == 4 * MiB
    assert "decode(encode(x)) == x for every Block" in ln["parity"]
    for k in ("metric", "value", "unit", "ms_per_step", "higher_is_better", "scaling", "dtype", "data", "roofline", "clocks", "gpu_launches"):
        assert k in ln


def test_dump_outputs(tmp_path):
    """--dump-outputs: the last timed step's Index records, per-Block SHA-256 and encoded bytes, as float arrays."""
    import hashlib
    import numpy as np
    _run(1, ["--dump-outputs", str(tmp_path)])
    recs = np.load(tmp_path / "index_records.npy")
    sha = np.load(tmp_path / "block_sha256.npy")
    blocks = np.load(tmp_path / "blocks_sample.npy")
    assert recs.dtype == np.float64 and recs.shape == (4, 2) and (recs[:, 1] == MiB).all()
    assert sha.dtype == np.float32 and sha.shape == (4, 32) and blocks.dtype == np.float32
    sizes = (recs[:, 0].astype(np.int64) + 3) // 4 * 4
    assert len(blocks) == sizes.sum()   # 4 MiB of input: all encoded bytes, no sample
    raw = blocks.astype(np.uint8).tobytes()
    offs = np.concatenate([[0], np.cumsum(sizes)])
    for i in range(4):
        assert hashlib.sha256(raw[offs[i]:offs[i + 1]]).digest() == sha[i].astype(np.uint8).tobytes()


def test_two_ranks_weak_scaling_job_is_per_gpu():
    """config 1 at N = 2: every rank takes the whole per-GPU job (4 Blocks here), the Stream has 8 records."""
    ln = _run(2, [])
    assert ln["scaling"] == "weak" and ln["n_gpus"] == 2
    assert ln["config"]["total_bytes"] == 8 * MiB and ln["index_records"] == 8
    assert ln["e2e"]["h2d_bytes_per_step"] == 8 * MiB and ln["decode"]["d2h_bytes_per_step"] == 8 * MiB
    assert "2 GPUs x 4 MiB (4 Blocks per GPU, weak scaling)" in ln["config"]["workload"]
    assert "ROUND TRIP FAILED" not in ln["parity"]


def test_two_ranks_strong_scaling_splits_the_job():
    ln = _run(2, ["--scaling", "strong"])
    assert ln["scaling"] == "strong" and ln["config"]["total_bytes"] == 4 * MiB and ln["index_records"] == 4
    assert ln["e2e"]["h2d_bytes_per_step"] == 4 * MiB
    assert "ROUND TRIP FAILED" not in ln["parity"]
