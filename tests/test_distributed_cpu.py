"""World-size-2 gloo tests (CPU) of the host logic of the multi-GPU path: shard ranges, the in-place
variable-length all-gather of per-rank edge blocks, and the rank-order exchange of the attribute
statistics.  The kernels themselves need a GPU; here the per-rank blocks are produced with numpy."""

import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from anemoi_graphs_b200 import device as agx_device


def _free_port() -> int:
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank: int, world: int, port: int, out_dir: str) -> None:
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        assert agx_device.world() == (rank, world)
        # a search is sharded only from SHARD_MIN_QUERIES query nodes; below it every rank does all of it
        assert agx_device.shard_world(agx_device.SHARD_MIN_QUERIES) == (rank, world)
        assert agx_device.shard_world(agx_device.SHARD_MIN_QUERIES - 1) == (0, 1) or agx_device.SHARD_MIN_QUERIES == 0
        # --- KNN-like fixed-size blocks: 11 queries x k=3 --------------------------------------------
        nq, k = 11, 3
        lo, hi = agx_device.shard_range(nq)
        full = torch.full((2, nq * k), -1, dtype=torch.int32)
        q = torch.arange(lo, hi, dtype=torch.int32).repeat_interleave(k)
        full[0, lo * k : hi * k] = 100 + q * 7 % 13
        full[1, lo * k : hi * k] = q
        counts = [(b - a) * k for a, b in (agx_device.shard_range(nq, r, world) for r in range(world))]
        agx_device.all_gather_v(full, counts, dim=1)
        allq = torch.arange(nq, dtype=torch.int32).repeat_interleave(k)
        assert torch.equal(full[1], allq) and torch.equal(full[0], 100 + allq * 7 % 13)
        # --- equal blocks (in-place all_gather_into_tensor path) -----------------------------------
        full = torch.full((2, 8), -1, dtype=torch.int32)
        full[:, rank * 4 : rank * 4 + 4] = torch.arange(4, dtype=torch.int32) + 10 * rank
        agx_device.all_gather_v(full, [4, 4], dim=1)
        assert full[0].tolist() == [0, 1, 2, 3, 10, 11, 12, 13] and torch.equal(full[0], full[1])
        # --- cut-off-like variable-size blocks ------------------------------------------------------
        mine = 5 if rank == 0 else 2
        counts = agx_device.all_gather_counts(mine, torch.device("cpu"))
        assert counts == [5, 2]
        full = torch.zeros((2, sum(counts)), dtype=torch.int32)
        off = sum(counts[:rank])
        full[:, off : off + mine] = rank + 1
        agx_device.all_gather_v(full, counts, dim=1)
        assert full[0].tolist() == [1] * 5 + [2] * 2 and full[1].tolist() == [1] * 5 + [2] * 2
        # --- asynchronous exchange: the other rank's block is complete after wait_for / flush -----------
        full = torch.zeros((2, sum(counts)), dtype=torch.int32)
        full[:, off : off + mine] = rank + 1
        agx_device.all_gather_v(full, counts, dim=1, async_op=True)
        side = torch.zeros((sum(counts), 1), dtype=torch.float32)
        side[off : off + mine] = float(rank + 1)
        agx_device.all_gather_v(side, counts, dim=0, async_op=True)
        agx_device.wait_for(full)
        assert full[0].tolist() == [1] * 5 + [2] * 2 and full[1].tolist() == [1] * 5 + [2] * 2
        agx_device.flush()  # waits for `side`
        assert side[:, 0].tolist() == [1.0] * 5 + [2.0] * 2
        # --- chunked exchange of uneven blocks (ChunkedGather): padded equal-block all-gathers per chunk, one chunk
        #     empty on one rank, one empty on both ---------------------------------------------------------------
        mine = [3, 0, 2, 0] if rank == 0 else [1, 4, 0, 0]
        rows = agx_device.all_gather_count_rows(mine, torch.device("cpu"))
        assert rows == [[3, 0, 2, 0], [1, 4, 0, 0]]
        full = torch.full((2, 10), -1, dtype=torch.int32)
        gather = agx_device.ChunkedGather(full, rows)
        assert gather.offsets == [[0, 3, 3, 5], [5, 6, 10, 10]]
        for c in range(4):
            o, n = gather.offsets[rank][c], rows[rank][c]
            full[0, o : o + n] = 100 * rank + 10 * c + torch.arange(n, dtype=torch.int32)  # "search" of chunk c
            full[1, o : o + n] = c
            gather.chunk_done(c, gather.mark())
        gather.finish()
        assert full[0].tolist() == [0, 1, 2, 20, 21, 100, 110, 111, 112, 113]
        assert full[1].tolist() == [0, 0, 0, 2, 2, 0, 1, 1, 1, 1]
        assert agx_device.query_chunks(10, 21, 3) == [(10, 13), (13, 17), (17, 21)]
        assert agx_device.n_query_chunks(100, 2) == 1
        # --- an empty rank block --------------------------------------------------------------------
        counts = agx_device.all_gather_counts(0 if rank == 1 else 4, torch.device("cpu"))
        full = torch.zeros((sum(counts), 2), dtype=torch.float32)
        if rank == 0:
            full[:4] = 3.5
        agx_device.all_gather_v(full, counts, dim=0)
        assert torch.equal(full, torch.full((4, 2), 3.5))
        # --- attribute statistics: sums add, minima / maxima combine, identical on every rank --------
        rng = np.random.default_rng(5)
        v = rng.random(1000)
        lo, hi = agx_device.shard_range(1000)
        part = v[lo:hi]
        st = torch.tensor([part.sum(), (part**2).sum(), part.min(), part.max()] * 2, dtype=torch.float64)
        raw = agx_device.all_gather_stats_raw(st)  # what the kernel folds, in rank order
        assert raw.shape == (world, 8) and torch.equal(raw[rank], st)
        np.testing.assert_allclose(raw[:, 0].sum().item(), v.sum(), rtol=1e-14)
        np.testing.assert_allclose(raw[:, 5].sum().item(), (v**2).sum(), rtol=1e-14)
        assert raw[:, 2].min().item() == v.min() and raw[:, 7].max().item() == v.max()
        # two sets per rank (the deferred decoder's): (W, 16), still rank-major
        two = agx_device.all_gather_stats_raw(torch.stack([st, 2 * st]))
        assert two.shape == (world, 16) and torch.equal(two[rank], torch.cat([st, 2 * st]))
        assert torch.equal(two[:, :8], raw)
        torch.save(raw, os.path.join(out_dir, f"stats{rank}.pt"))
        dist.barrier()
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(120)
def test_two_rank_gather_and_statistics_tables(tmp_path):
    port = _free_port()
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    a, b = torch.load(tmp_path / "stats0.pt"), torch.load(tmp_path / "stats1.pt")
    assert torch.equal(a, b)  # bitwise identical statistics tables, so identical constants, on every rank
