"""Checkpoint bookkeeping without a GPU: merging the state dicts of several shards, picking one shard's records, and the
refusals that happen before any library call."""
import pytest
import torch

from wab_gym_b200.sharding import merge_state_dicts, select_shard_records, shard_range

R = 32     # record width used here (the real one comes from the library; these functions only move rows)


def _sd(first, count, fp=7, fmt=1, stats=None):
    ids = torch.arange(first, first + count, dtype=torch.int64)
    records = (ids[:, None] * 3 + torch.arange(R)[None, :]).to(torch.uint8)     # row content identifies its id
    return {"format": fmt, "fingerprint": fp, "env_ids": ids, "records": records,
            "stats": torch.tensor(stats if stats is not None else [first] * 8, dtype=torch.int64)}


def _row(i):
    return (torch.tensor(i) * 3 + torch.arange(R)).to(torch.uint8)


@pytest.mark.parametrize("total,old_world,new_world", [(1000, 1, 3), (1000, 8, 2), (37, 3, 5), (10, 4, 4), (7, 2, 7)])
def test_reshard_selects_every_id_once_in_slot_order(total, old_world, new_world):
    parts = [_sd(*shard_range(total, r, old_world)) for r in range(old_world)]
    merged = merge_state_dicts(parts[::-1])                # order of the ranks does not matter
    assert merged["records"].shape == (total, R)
    assert merged["stats"].tolist() == [sum(shard_range(total, r, old_world)[0] for r in range(old_world))] * 8
    seen = []
    for r in range(new_world):
        first, count = shard_range(total, r, new_world)
        rec = select_shard_records(merged, first, count, 7, R)
        assert rec.shape == (count, R)
        for s in range(count):
            assert torch.equal(rec[s], _row(first + s))
        seen.extend(range(first, first + count))
    assert seen == list(range(total))


def test_missing_or_duplicated_ids_are_refused():
    sd = merge_state_dicts([_sd(0, 5), _sd(6, 4)])       # id 5 missing
    with pytest.raises(ValueError, match="no record"):
        select_shard_records(sd, 0, 10, 7, R)
    assert select_shard_records(sd, 6, 4, 7, R).shape == (4, R)
    dup = merge_state_dicts([_sd(0, 5), _sd(3, 5)])      # ids 3, 4 twice
    with pytest.raises(ValueError, match="more than one"):
        select_shard_records(dup, 0, 8, 7, R)
    assert select_shard_records(dup, 5, 3, 7, R).shape == (3, R)


def test_format_fingerprint_and_width_mismatches_are_refused():
    with pytest.raises(ValueError, match="format"):
        select_shard_records(_sd(0, 4, fmt=2), 0, 4, 7, R)
    with pytest.raises(ValueError, match="fingerprint"):
        select_shard_records(_sd(0, 4, fp=8), 0, 4, 7, R)
    with pytest.raises(ValueError, match="records must be"):
        select_shard_records(_sd(0, 4), 0, 4, 7, R + 16)
    with pytest.raises(ValueError):
        merge_state_dicts([_sd(0, 4), _sd(4, 4, fp=9)])
    with pytest.raises(ValueError):
        merge_state_dicts([])


def test_state_entry_points_are_declared_and_exported():
    from wab_gym_b200 import _lib
    for name in ("wab_vec_state_record_bytes", "wab_vec_state_fingerprint", "wab_vec_save_state", "wab_vec_load_state",
                 "wab_vec_set_stats"):
        assert name in _lib.EXPORTS
        assert hasattr(_lib.load(), name)
