"""GPU, world_size 2 (skipped on a one-GPU box): BASELINE.json config 5's pass criterion — the match tables gathered over NCCL are
bit-equal to the single-GPU run.  bench.py runs the same 64-pair job at every N (`table_check`: contiguous blocks of frames + one
halo frame per rank, extraction, matching, one all-gather) and prints a checksum of the gathered table; here N = 1 and N = 2 are
launched the way the driver launches them and their checksums compared.  (The host-side sharding logic is covered on CPU with
gloo in tests/test_batch_cpu.py.)"""
import json
import os
import subprocess
import sys
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu


def _run(n):
    env = dict(os.environ, SSLPL_BENCH_NO_TRACE="1")
    base = [os.path.join(ROOT, "bench.py"), "--gpus", str(n), "--steps", "2", "--warmup", "3", "--no-cpu-baseline", "--scaling", "strong"]
    cmd = [sys.executable] + base if n == 1 else [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
                                                   "--master-addr", "127.0.0.1", "--master-port", "29541"] + base
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("{")][-1]
    return json.loads(line)


def test_gathered_tables_equal_single_gpu():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    a, b = _run(1), _run(2)
    assert a["table_check"]["rows"] == b["table_check"]["rows"] == 64 and a["table_check"]["matches"] > 1000
    assert a["table_check"] == {**b["table_check"], "frames": a["table_check"]["frames"]} or a["table_check"]["checksum"] == b["table_check"]["checksum"], (a["table_check"], b["table_check"])
    assert a["table_check"]["checksum"] == b["table_check"]["checksum"] and a["table_check"]["matches"] == b["table_check"]["matches"]
    assert b["gather_check"]["ok_on_every_rank"] and b["n_gpus"] == 2 and b["scaling"] == "strong"
