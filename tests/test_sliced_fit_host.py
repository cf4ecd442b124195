"""Host (CPU) tests of the pixel-sliced fit step: slice plan, rank -> slice mapping, schedule parsing, and the
gather-and-sum orchestration on a gloo world of 2 with a CPU stand-in for the native row producer."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from awesome_b200.fit import gather_slice_rows, rank_slices, slice_plan
from awesome_b200.pretrain import FitSchedule


@pytest.mark.parametrize("n", [1, 5, 127, 128, 129, 1000, 4095, 2 * 640 * 480, 6 * 48 * 64])
@pytest.mark.parametrize("S", [1, 3, 4, 8])
def test_slice_plan_covers_rows_with_aligned_balanced_slices(n, S):
    plan = slice_plan(n, S)
    assert len(plan) == S
    assert plan[0][0] == 0 and plan[-1][1] == n
    for (b0, e0), (b1, _) in zip(plan, plan[1:]):
        assert e0 == b1                                  # contiguous, in order
    for b, e in plan:
        assert b <= e
        assert b % 128 == 0 and (e % 128 == 0 or e == n)
    sizes = [e - b for b, e in plan]
    assert max(sizes) - min(sizes) <= 128


def test_slice_plan_small_batches_and_errors():
    assert slice_plan(5, 8)[-1] == (0, 5) and all(b == e for b, e in slice_plan(5, 8)[:-1])   # N < S: one live slice
    assert [e - b for b, e in slice_plan(300, 4)] == [0, 128, 128, 44]
    assert slice_plan(2 * 640 * 480, 8)[0] == (0, 76800)
    with pytest.raises(ValueError):
        slice_plan(0, 4)
    with pytest.raises(ValueError):
        slice_plan(10, 0)


def test_rank_slices_mapping():
    assert list(rank_slices(8, 0, 1)) == list(range(8))
    assert [list(rank_slices(8, r, 2)) for r in range(2)] == [[0, 1, 2, 3], [4, 5, 6, 7]]
    assert [list(rank_slices(8, r, 8)) for r in range(8)] == [[r] for r in range(8)]
    for world in (1, 2, 4, 8):
        owned = [k for r in range(world) for k in rank_slices(8, r, world)]
        assert owned == list(range(8))
    with pytest.raises(ValueError, match="multiple"):
        rank_slices(8, 0, 3)
    with pytest.raises(ValueError):
        rank_slices(8, 2, 2)


def test_schedule_parses_sequence_slices():
    assert FitSchedule().sequence_slices == 0
    s = FitSchedule.from_pretrain_args({"sequence_slices": 8, "batch_size": 2, "unknown_arg": 1})
    assert s.sequence_slices == 8 and s.batch_size == 2


def _stand_in_row(k: int, step: int, R: int) -> torch.Tensor:
    # distinct, non-associative-friendly values per slice and step
    g = torch.Generator().manual_seed(1000 * step + k)
    return torch.randn(R, generator=g) * (10.0 ** (k % 3))


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        S, R, P = 8, 9, 8
        mine = rank_slices(S, rank, world)
        rows = torch.zeros(S, R)
        local = torch.zeros(len(mine), R)
        params = torch.zeros(P)
        ok = True
        for step in range(3):
            produced = []

            def produce(k, row, j):
                produced.append((k, j))
                row.copy_(_stand_in_row(k, step, R))

            got = gather_slice_rows(mine, local, rows, produce)
            ok &= produced == [(k, j) for j, k in enumerate(mine)]
            # rows arrive in slice order, bit for bit
            ok &= all(torch.equal(got[k], _stand_in_row(k, step, R)) for k in range(S))
            # stand-in optimizer: sum in row order, then a step
            g = torch.zeros(R)
            for k in range(S):
                g += got[k]
            params -= 0.1 * g[:P]
        allp = [torch.zeros(P) for _ in range(world)]
        dist.all_gather(allp, params)
        same = all(torch.equal(allp[0], p) for p in allp)
        flag = torch.tensor([1.0 if ok and same else 0.0])
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if rank == 0:
            # the one-rank run of the same orchestration gives the same parameters
            rows1 = torch.zeros(S, R)
            p1 = torch.zeros(P)
            for step in range(3):
                got = gather_slice_rows(range(S), rows1, rows1, lambda k, row, j: row.copy_(_stand_in_row(k, step, R)))
                g = torch.zeros(R)
                for k in range(S):
                    g += got[k]
                p1 -= 0.1 * g[:P]
            out.put((float(flag), torch.equal(p1, params)))
    finally:
        dist.destroy_process_group()


def test_gather_and_sum_world2_gloo():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    assert q.get(timeout=10) == (1.0, True)
