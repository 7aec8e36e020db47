"""N>1 host logic on CPU: world_size-2 gloo run of the sharding helpers used by bench.py --gpus N."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

WORKER = r'''
import os, sys
sys.path.insert(0, sys.argv[1])
import torch, torch.distributed as dist
from fhe_rs_b200.shard import shard_range, max_over_ranks, gather_checksums
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
total = 11
first, last = shard_range(total, rank, world)
local = [(7919 * i + 13) % (1 << 40) for i in range(first, last)]      # stand-in per-ciphertext checksums
allc = gather_checksums(local)
assert allc == [(7919 * i + 13) % (1 << 40) for i in range(total)], allc
t = max_over_ranks(1.0 + rank)
assert t == float(world), t
dist.barrier()
if rank == 0:
    print("SHARD_OK", first, last, len(allc))
dist.destroy_process_group()
'''


def test_shard_range_properties():
    sys.path.insert(0, ROOT)
    from fhe_rs_b200.shard import shard_range
    for total in (0, 1, 7, 64, 65536, 1000):
        for world in (1, 2, 3, 4, 8):
            blocks = [shard_range(total, r, world) for r in range(world)]
            assert blocks[0][0] == 0 and blocks[-1][1] == total
            for a, b in zip(blocks, blocks[1:]):
                assert a[1] == b[0]
            sizes = [b - a for a, b in blocks]
            assert max(sizes) - min(sizes) <= 1


def test_two_rank_gloo(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    # --standalone: a local rendezvous on a free port, so that concurrent runs on one host do not collide
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--standalone", "--nproc-per-node=2",
                          str(script), ROOT], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "SHARD_OK" in out.stdout, out.stdout + out.stderr


def test_numa_binding_never_raises():
    """bind_host_thread_to_gpu is an optimisation for the end-to-end path: without a GPU / NVML it must report that it
    did nothing instead of raising"""
    from fhe_rs_b200.shard import bind_host_thread_to_gpu
    msg = bind_host_thread_to_gpu(0)
    assert isinstance(msg, str) and msg
