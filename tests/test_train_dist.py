"""Host side of data-parallel training on CPU: shard validation, minibatch counts, seed folding, merged trainer
checkpoints, and the rank-order sums of a world-size-2 gloo run."""
import os
import socket

import pytest
import torch
import torch.multiprocessing as mp

from wab_gym_b200.sharding import (check_trainer_shards, global_mean_std, global_minibatch_counts, merge_trainer_state_dicts,
                                   minibatch_bounds, rank_order_sum, shard_range)


def test_shards_must_tile_the_batch_in_rank_order_and_agree():
    sig = (0xABC, 5, 64, "horizon", 0.99)
    assert check_trainer_shards([(f, c, sig) for f, c in (shard_range(1001, r, 3) for r in range(3))]) == 1001
    assert check_trainer_shards([(0, 7, sig)]) == 7
    for bad in ([(0, 500, sig), (501, 500, sig)],          # a gap
                [(0, 500, sig), (499, 500, sig)],          # an overlap
                [(500, 500, sig), (0, 500, sig)],          # out of rank order
                [(1, 500, sig)],                           # not starting at 0
                [(0, 500, sig), (500, 0, sig)],            # an empty shard
                [(0, 500, sig), (500, 500, sig[:-1] + (0.9,))]):   # another hyper-parameter
        with pytest.raises(ValueError):
            check_trainer_shards(bad)


def test_minibatch_bounds_and_global_counts_for_ragged_shards():
    assert minibatch_bounds(10, 4) == [0, 2, 5, 7, 10]
    T, total, world, mb = 16, 1003, 3, 4
    rows = [T * shard_range(total, r, world)[1] for r in range(world)]
    counts = global_minibatch_counts(rows, mb)
    assert sum(counts) == T * total
    for k in range(mb):
        assert counts[k] == sum(minibatch_bounds(r, mb)[k + 1] - minibatch_bounds(r, mb)[k] for r in rows)
    # one rank: the trainer's own counts
    assert global_minibatch_counts([T * total], mb) == [b - a for a, b in zip(minibatch_bounds(T * total, mb), minibatch_bounds(T * total, mb)[1:])]


def test_permutation_seed_folds_the_shard_only_when_distributed():
    from wab_gym_b200.ppo import _perm_seed, _seed
    assert _perm_seed(123, 4, 1) == _seed(123, 4, 1)                    # group=None: the single-process seed
    assert _perm_seed(123, 4, 1, 0) == _seed(123, 4, 1, 0) != _seed(123, 4, 1)
    assert len({_perm_seed(123, 4, 1, b) for b in (0, 500, 1000)}) == 3


def _trainer_sd(first, count, scale=1.0, ctr=7, extra=None):
    sd = {"env": {"format": 1, "fingerprint": 99, "env_ids": torch.arange(first, first + count),
                  "records": torch.full((count, 16), first, dtype=torch.uint8), "stats": torch.arange(8)},
          "policy": {"w": torch.tensor([1.0, -0.0, scale])},
          "optimizer": {"state": {0: {"step": torch.tensor(3.0), "exp_avg": torch.ones(3)}}, "param_groups": [{"lr": 3e-4, "params": [0]}]},
          "noise_ctr": ctr, "sample_seed": 5, "iteration": 2}
    if extra:
        sd.update(extra)
    return sd


def test_merge_trainer_state_dicts_joins_envs_and_checks_shared_parts():
    m = merge_trainer_state_dicts([_trainer_sd(0, 3), _trainer_sd(3, 2)])
    assert m["env"]["env_ids"].tolist() == [0, 1, 2, 3, 4] and m["env"]["records"].shape == (5, 16)
    assert m["env"]["stats"].tolist() == [2 * i for i in range(8)]
    assert m["noise_ctr"] == 7 and m["iteration"] == 2 and torch.equal(m["policy"]["w"], torch.tensor([1.0, -0.0, 1.0]))
    for other in (_trainer_sd(3, 2, scale=1.0 + 2 ** -20), _trainer_sd(3, 2, ctr=8), _trainer_sd(3, 2, extra={"iteration": 3}),
                  _trainer_sd(3, 2, extra={"policy": {"w": torch.tensor([1.0, 0.0, 1.0])}}),          # -0.0 vs 0.0: not bit-equal
                  _trainer_sd(3, 2, extra={"optimizer": {"state": {0: {"step": torch.tensor(4.0), "exp_avg": torch.ones(3)}},
                                                         "param_groups": [{"lr": 3e-4, "params": [0]}]}})):
        with pytest.raises(ValueError):
            merge_trainer_state_dicts([_trainer_sd(0, 3), other])
    with pytest.raises(ValueError):
        merge_trainer_state_dicts([])


def _worker(rank, world, port, out):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    g = torch.Generator().manual_seed(1)
    full = torch.randn(1003, generator=g) * 3 + 1
    first, count = shard_range(full.numel(), rank, world)
    mean, std = global_mean_std(full[first:first + count])
    s = rank_order_sum(torch.tensor([0.1 * (rank + 1), 1e16, -1e16], dtype=torch.float64))
    out[rank] = (float(mean), float(std), s.tolist())
    dist.barrier()
    dist.destroy_process_group()


def test_rank_order_statistics_gloo_world_size_2():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_worker, args=(2, port, out), nprocs=2, join=True)
    assert out[0] == out[1]                                                   # the same bits on every rank
    g = torch.Generator().manual_seed(1)
    full = (torch.randn(1003, generator=g) * 3 + 1).double()
    mean = full.sum() / full.numel()
    assert out[0][0] == float(mean.float())
    assert abs(out[0][1] - float(full.std())) <= 1e-6 * float(full.std())
    assert out[0][2] == [0.1 + 0.2, 1e16 + 1e16, -1e16 + -1e16]               # rank 0 first, then rank 1
