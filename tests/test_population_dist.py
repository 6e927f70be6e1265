"""Host side of data-parallel populations on CPU: the shard layout and its refusals, the blocked-id arithmetic, the
members' global normalisation statistics and merged population checkpoints, and the constructor refusals raised on every
rank of a world-size-2 gloo group."""
import os
import socket

import pytest
import torch
import torch.multiprocessing as mp

from wab_gym_b200.sharding import (blocked_env_ids, blocked_env_slots, check_population_shards, global_mean_std,
                                   global_mean_std_members, merge_population_state_dicts, population_shards, shard_range)


def _port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def test_population_shards_are_shard_range_in_multiples_of_128():
    assert population_shards(2048, 1) == [(0, 2048)]
    assert population_shards(2048, 8) == [(256 * r, 256) for r in range(8)]
    assert population_shards(640, 5) == [shard_range(640, r, 5) for r in range(5)] == [(128 * r, 128) for r in range(5)]
    for n, world in ((1000, 2), (640, 2), (128, 2), (256, 3), (0, 1), (384, 4)):
        with pytest.raises(ValueError, match="multiple of 128"):
            population_shards(n, world)


def test_blocked_ids_against_a_loop():
    for blocks, c, stride, base in ((1, 384, 0, 0), (1, 256, 0, 77), (3, 128, 1000, 5), (4, 256, 256, 0), (2, 128, 0, 9)):
        rows = torch.arange(blocks * c)
        want = [base + (r // c) * stride + r % c for r in range(blocks * c)]
        ids = blocked_env_ids(rows, blocks, c, stride, base)
        assert ids.dtype == torch.int64 and ids.tolist() == want
        if stride == 0 and blocks > 1:
            continue                                        # replicas: ids repeat and have no inverse
        perm = torch.randperm(rows.numel(), generator=torch.Generator().manual_seed(blocks))
        assert torch.equal(blocked_env_slots(ids[perm], blocks, c, stride, base), rows[perm])
    # ids a handle does not hold: before its base, in the gap between blocks, past its last block
    for bad in (4, 5 + 128, 5 + 999, 5 + 3000):
        with pytest.raises(ValueError, match="outside"):
            blocked_env_slots(torch.tensor([5, bad]), 3, 128, 1000, 5)
    with pytest.raises(ValueError, match="outside"):
        blocked_env_slots(torch.tensor([77 + 256]), 1, 256, 0, 77)


def _info(base, num, blocks, stride, sig=("fp", 5)):
    return (base, num, blocks, stride, sig)


def test_population_layout_check():
    P, n = 3, 640
    layout = [(0, 384), (384, 256)]                         # any tiling in multiples of 128, not only population_shards'
    infos = [_info(f, P * c, P, n) for f, c in layout]
    assert check_population_shards(infos, P) == (0, n)
    shifted = [_info(1000 + f, P * c, P, n) for f, c in layout]
    assert check_population_shards(shifted, P) == (1000, n)
    assert check_population_shards([_info(0, 256, 1, 0)], 1) == (0, 256)       # one member: a plain handle
    assert check_population_shards([_info(0, 256, 1, 0), _info(256, 128, 1, 0)], 1) == (0, 384)
    for bad, match in (([_info(0, 3 * 384, 3, 640), _info(385, 3 * 256, 3, 640)], "tile"),          # a gap
                       ([_info(0, 3 * 384, 3, 640), _info(383, 3 * 256, 3, 640)], "tile"),          # an overlap
                       ([_info(384, 3 * 256, 3, 640), _info(0, 3 * 384, 3, 640)], "tile"),          # out of rank order
                       ([_info(0, 3 * 384, 3, 640), _info(384, 3 * 256, 3, 384)], "block_stride"),
                       ([_info(0, 3 * 384, 1, 0), _info(384, 3 * 256, 3, 640)], "blocks"),
                       ([_info(0, 3 * 384, 3, 640), _info(384, 3 * 200, 3, 640)], "multiple of 128"),
                       ([_info(0, 3 * 384, 3, 640), _info(384, 2 * 256, 3, 640)], "multiple of 128"),
                       ([_info(0, 3 * 384, 3, 640), _info(384, 3 * 256, 3, 640, ("fp", 6))], "differs")):
        with pytest.raises(ValueError, match=match):
            check_population_shards(bad, 3)


def _pop_sd(first, count, members=2, n=256, scale=1.0, ctr=7, lr=3e-4):
    ids = torch.cat([torch.arange(p * n + first, p * n + first + count) for p in range(members)])
    return {"env": {"format": 1, "fingerprint": 99, "env_ids": ids, "records": ids[:, None].repeat(1, 16).to(torch.uint8),
                    "stats": torch.arange(8)},
            "policies": [{"w": torch.tensor([1.0, -0.0, scale * (p + 1)])} for p in range(members)],
            "optimizers": [{"state": {0: {"step": torch.tensor(3.0), "exp_avg": torch.ones(3)}},
                            "param_groups": [{"lr": lr, "params": [0]}]} for _ in range(members)],
            "hyperparameters": [{"lr": lr, "gamma": 0.99} for _ in range(members)], "noise_ctr": ctr, "sample_seed": 5,
            "iteration": 2}


def test_merge_population_state_dicts_round_trip_and_refusals():
    from wab_gym_b200.sharding import select_shard_records
    parts = [_pop_sd(0, 128), _pop_sd(128, 128)]
    m = merge_population_state_dicts(parts)
    assert sorted(m["env"]["env_ids"].tolist()) == list(range(512))
    assert m["env"]["stats"].tolist() == [2 * i for i in range(8)]
    assert m["iteration"] == 2 and m["noise_ctr"] == 7 and m["hyperparameters"] == parts[0]["hyperparameters"]
    assert all(torch.equal(a["w"], b["w"]) for a, b in zip(m["policies"], parts[0]["policies"]))
    # each member's contiguous id range comes back out of the merged dict, in slot order, on any layout
    for p in range(2):
        rec = select_shard_records(m["env"], p * 256, 256, 99, 16)
        assert torch.equal(rec[:, 0], torch.arange(p * 256, (p + 1) * 256).to(torch.uint8))
    for other in (_pop_sd(128, 128, scale=1.0 + 2 ** -20), _pop_sd(128, 128, ctr=8), _pop_sd(128, 128, lr=1e-3)):
        with pytest.raises(ValueError, match="differs"):
            merge_population_state_dicts([parts[0], other])
    with pytest.raises(ValueError):
        merge_population_state_dicts([])


def _stats_worker(rank, world, port, out):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    g = torch.Generator().manual_seed(2)
    full = torch.randn(3, 16, 768, generator=g) * torch.tensor([1.0, 3.0, 0.1])[:, None, None] + 2
    first, c = [(0, 512), (512, 256)][rank]                         # a ragged layout
    mine = full[:, :, first:first + c].contiguous()                 # [P, T, c]: every member's shard on this rank
    mean, std = global_mean_std_members(mine)
    each = [global_mean_std(mine[p].contiguous()) for p in range(3)]
    out[rank] = (mean.tolist(), std.tolist(), [float(m) for m, _ in each], [float(s) for _, s in each])
    dist.barrier()
    dist.destroy_process_group()


def test_members_statistics_equal_per_member_global_mean_std_gloo():
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_stats_worker, args=(2, _port(), out), nprocs=2, join=True)
    assert out[0] == out[1]
    mean, std, want_mean, want_std = out[0]
    assert mean == want_mean and std == want_std                    # bit-equal (floats from fp32 scalars)


class _Env:
    """What the population's constructor reads before it touches a device (an env that raises on any other use)."""

    def __init__(self, num_envs, env_id_base=0, blocks=1, block_stride=0, with_features=True, fingerprint=0xF00):
        self.num_envs, self.env_id_base, self.blocks, self.block_stride = num_envs, env_id_base, blocks, block_stride
        self.with_features, self.fingerprint, self.flat_dim, self.n_actions = with_features, fingerprint, 449, 5

    @property
    def device(self):
        raise AssertionError("PPOPopulation touched the device before refusing")


# per case: the kwargs of rank 0 and of rank 1 (P = 2 members of n = 512 envs: c = 256 per rank)
_REFUSALS = [
    ("rank 1 not blocked", dict(env=dict(num_envs=512, blocks=2, block_stride=512)), dict(env=dict(num_envs=512, env_id_base=256)), "blocks"),
    ("gap", dict(env=dict(num_envs=512, blocks=2, block_stride=512)),
     dict(env=dict(num_envs=512, env_id_base=384, blocks=2, block_stride=512)), "tile"),
    ("stride", dict(env=dict(num_envs=512, blocks=2, block_stride=1024)),
     dict(env=dict(num_envs=512, env_id_base=256, blocks=2, block_stride=1024)), "block_stride"),
    ("ragged", dict(env=dict(num_envs=512, blocks=2, block_stride=640)),
     dict(env=dict(num_envs=2 * 192, env_id_base=256, blocks=2, block_stride=640)), "multiple of 128"),
    ("features", dict(env=dict(num_envs=512, blocks=2, block_stride=512)),
     dict(env=dict(num_envs=512, env_id_base=256, blocks=2, block_stride=512, with_features=False)), "features"),
    ("options", dict(env=dict(num_envs=512, blocks=2, block_stride=512)),
     dict(env=dict(num_envs=512, env_id_base=256, blocks=2, block_stride=512, fingerprint=0xF01)), "differs"),
    ("hyper-parameters", dict(env=dict(num_envs=512, blocks=2, block_stride=512)),
     dict(env=dict(num_envs=512, env_id_base=256, blocks=2, block_stride=512), hyperparameters=[{}, {"lr": 1e-3}]), "differs"),
    ("epochs", dict(env=dict(num_envs=512, blocks=2, block_stride=512)),
     dict(env=dict(num_envs=512, env_id_base=256, blocks=2, block_stride=512), epochs=2), "differs"),
    ("not a Policy", dict(env=dict(num_envs=512, blocks=2, block_stride=512)),
     dict(env=dict(num_envs=512, env_id_base=256, blocks=2, block_stride=512), policies=[object(), object()]), "rank 1"),
    ("bad hyper-parameter", dict(env=dict(num_envs=512, blocks=2, block_stride=512), hyperparameters=[{}, {"clip_eps": 0.0}]),
     dict(env=dict(num_envs=512, env_id_base=256, blocks=2, block_stride=512)), "clip_eps"),
]


def _refusal_worker(rank, world, port, out):
    import torch.distributed as dist
    from wab_gym_b200.population import PPOPopulation
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    res = []
    for name, kw0, kw1, match in _REFUSALS:
        kw = dict(kw0 if rank == 0 else kw1)
        env = _Env(**kw.pop("env"))
        try:
            PPOPopulation(env, 2, group=dist.group.WORLD, **kw)
            res.append((name, None))
        except ValueError as exc:
            res.append((name, str(exc)))
    out[rank] = res
    dist.barrier()
    dist.destroy_process_group()


def test_constructor_refusals_are_raised_on_every_rank_gloo():
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_refusal_worker, args=(2, _port(), out), nprocs=2, join=True)
    for r in range(2):
        for (name, _, _, match), (got_name, msg) in zip(_REFUSALS, out[r]):
            assert got_name == name and msg is not None and match in msg, (r, name, msg)


def test_a_group_without_torch_distributed_is_refused():
    from wab_gym_b200.population import PPOPopulation
    with pytest.raises(ValueError, match="group"):
        PPOPopulation(_Env(512), 2, group=object())
