"""bench.py's reference arm runs on the host cores and prints the contract's JSON line."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "1", "--fibres", "120"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "edges/s" and line["higher_is_better"] is True
    # the unmodified reference Block when its sources are on this box (/root/reference or the copy build() vendors under
    # baseline/_ref/), else the oracle port
    from oracle import ref_loader
    want = "reference" if ref_loader.reference_available() else "port"
    assert line["value"] > 0 and line["cpu_baseline"]["kind"] == want and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"] == {"value": line["value"], "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_can_be_forced_to_the_port():
    env = dict(os.environ, PFS_CPU_ARM="port")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "1", "--fibres", "120"], capture_output=True, text=True, timeout=300, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.loads(out.stdout.strip().splitlines()[-1])["cpu_baseline"]["kind"] == "port"


def _teardown_worker(rank, world, port):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    sys.path.insert(0, ROOT)
    import bench
    import torch
    t = torch.ones(3)
    dist.all_reduce(t)
    assert float(t[0]) == world
    bench.shutdown_process_group()           # returns (the watchdog is cancelled) and leaves no initialised group behind
    assert not dist.is_initialized()


def test_process_group_teardown_returns_on_every_rank():
    import socket
    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_teardown_worker, args=(2, port), nprocs=2, join=True)
