"""CPU, world_size 2, gloo: the multi-rank host logic (ray sharding on chunk boundaries + gather back to frame order)."""
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_shard_ranges_partition_on_chunk_boundaries():
    from neo360_b200.sharding import shard_range
    for n, world, chunk in ((307200, 8, 1024), (1728, 2, 512), (1000, 4, 1024), (5, 2, 0), (1281 * 961, 8, 1024)):
        ranges = [shard_range(n, world, r, chunk) for r in range(world)]
        assert ranges[0][0] == 0 and ranges[-1][1] == n
        for (a, b), (c, d) in zip(ranges[:-1], ranges[1:]):
            assert b == c and a <= b
        for a, b in ranges:
            if chunk > 0 and b < n:
                assert a % chunk == 0 and b % chunk == 0      # quirk Q1: never split a chunk


def _worker(rank, world, port, n, chunk, tmp):
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    from neo360_b200.sharding import shard_batch, gather_rays
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    g = torch.Generator().manual_seed(0)
    batch = {"rays_o": torch.rand(n, 3, generator=g), "rays_d": torch.rand(n, 3, generator=g), "viewdirs": torch.rand(n, 3, generator=g),
             "src_poses": torch.eye(4).repeat(3, 1, 1), "target": torch.rand(n, 3, generator=g)}
    local, (a, b) = shard_batch(batch, world, rank, chunk)
    assert local["src_poses"].shape == (3, 4, 4) and local["rays_o"].shape[0] == b - a and local["target"].shape[0] == b - a
    # stand-in for the per-rank render: a per-ray function of the inputs
    rgb = local["rays_o"] * 2 + local["rays_d"]
    full = gather_rays(rgb, n, world, chunk)
    assert torch.equal(full, batch["rays_o"] * 2 + batch["rays_d"])
    dist.barrier()
    dist.destroy_process_group()
    open(os.path.join(tmp, f"ok{rank}"), "w").write("ok")


@pytest.mark.parametrize("n,chunk", [(1728, 512), (1000, 1024), (4096, 1024)])
def test_two_rank_gloo_shard_and_gather(tmp_path, n, chunk):
    import socket
    import torch.multiprocessing as mp
    s = socket.socket()                  # a port the OS reports free, not a fixed one another process may hold
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    mp.spawn(_worker, args=(2, port, n, chunk, str(tmp_path)), nprocs=2, join=True)
    assert (tmp_path / "ok0").exists() and (tmp_path / "ok1").exists()
