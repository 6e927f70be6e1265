"""Checkpoint, resume and clone on the device: a resumed run equals the run that never stopped, byte for byte, on every
kernel family, on any shard layout; clones share their source's world; refused loads change nothing."""
import copy
import ctypes
import pickle

import numpy as np
import pytest
import torch

from tests.util import OPTION_SETS

pytestmark = pytest.mark.gpu

K1, K2 = 37, 70


def _vec(*a, **k):
    from wab_gym_b200 import VecEnv
    return VecEnv(*a, **k)


def _acts(seed, steps, n, n_actions=5):
    rng = np.random.default_rng(seed)
    return torch.from_numpy(rng.integers(0, n_actions, size=(steps, n)).astype(np.uint8)).cuda()


def _host(obs, reward=None, done=None, info=None, features=None):
    out = {k: getattr(obs, k) for k in ("grids", "food", "role", "status")}
    out.update(reward=reward, done=done, info=info, features=features)
    return {k: v.detach().cpu().numpy().copy() for k, v in out.items() if v is not None}


def _run(env, acts, many=False):
    """Every output of len(acts) steps, one dict per step (or per launch with many=True)."""
    if many:
        o, r, d, i = env.step_many(acts)
        return [_host(o, r, d, i["info"], i.get("features"))]
    res = []
    for a in acts:
        o, r, d, i = env.step(a)
        res.append(_host(o, r, d, i["info"], i.get("features")))
    return res


def _same(a, b, what=""):
    assert len(a) == len(b)
    for t, (x, y) in enumerate(zip(a, b)):
        assert x.keys() == y.keys()
        for k in x:
            assert np.array_equal(x[k], y[k]), (what, t, k)


def _same_state(sa, sb):
    for k in sa:
        assert np.array_equal(sa[k], sb[k]), k


def _resume_equals_uninterrupted(tmp_path, n, kw, many=False, ego=False, n_actions=5):
    acts = _acts(11, K1 + K2, n, n_actions)
    a = _vec(n, seed=3, ego=ego, **kw)
    a.reset()
    head = _run(a, acts[:K1], many)
    tail = _run(a, acts[K1:], many)
    b = _vec(n, seed=3, ego=ego, **kw)
    b.reset()
    head_b = _run(b, acts[:K1], many)
    _same(head, head_b)
    ego_b = b.ego_proximities().cpu().numpy() if ego else None
    torch.save(b.state_dict(), tmp_path / "ckpt.pt")
    b.close()
    c = _vec(n, seed=3, ego=ego, **kw)
    c.reset()
    sd = torch.load(tmp_path / "ckpt.pt")
    obs = c.load_state_dict(sd)
    last = {k: (v[-1] if many else v) for k, v in head[-1].items()}
    reemitted = _host(obs, features=c.last_features)
    for k, v in reemitted.items():                         # the load returns what the last step returned
        assert np.array_equal(v, last[k]), k
    if ego:
        assert np.array_equal(c.ego_proximities().cpu().numpy(), ego_b)
    assert torch.equal(c.save_state().records.cpu(), sd["records"])      # save -> load -> save is byte-identical
    _same(tail, _run(c, acts[K1:], many), "tail")
    _same_state(a.export_state(), c.export_state())
    assert a.stats() == c.stats()
    if ego:
        assert np.array_equal(a.ego_proximities().cpu().numpy(), c.ego_proximities().cpu().numpy())
    a.close(); c.close()


@pytest.mark.parametrize("name", sorted(OPTION_SETS))
def test_resume_equals_uninterrupted_option_sets(tmp_path, name):
    from wab_gym_b200.config import GameConfig
    overrides = OPTION_SETS[name][0]
    na = GameConfig.from_options(overrides).n_actions
    _resume_equals_uninterrupted(tmp_path, 37, dict(game_options=overrides, features=True), n_actions=na)


@pytest.mark.parametrize("f64", [False, True])
@pytest.mark.parametrize("lpe", [1, 4, 8, 16, 32])
def test_resume_every_lanes_per_env_and_food_mode(tmp_path, monkeypatch, lpe, f64):
    monkeypatch.setenv("WAB_LPE", str(lpe))
    kw = dict(game_options={"chance_wolf_on_square": 0.01}, features=True, force_f64_food=f64)
    env = _vec(8, **kw)
    assert env.lanes_per_env == lpe and env.game.food_mode == (0 if f64 else 1)
    env.close()
    _resume_equals_uninterrupted(tmp_path, 100, kw)


def test_resume_two_warp_pipeline(tmp_path, monkeypatch):
    monkeypatch.setenv("WAB_PIPE", "2")
    monkeypatch.setenv("WAB_LPE", "8")
    _resume_equals_uninterrupted(tmp_path, 300, dict(game_options={"chance_wolf_on_square": 0.01}, features=True), many=True)


@pytest.mark.parametrize("geom", [(7, 9, 1), (15, 13, 2), (11, 11, 1)])
def test_resume_generic_kernels(tmp_path, monkeypatch, geom):
    W, H, m = geom
    if (W, H) == (11, 11):
        monkeypatch.setenv("WAB_GENERIC", "1")
    opts = {"width": W, "height": H, "wolf_spawn_margin": m, "chance_wolf_on_square": 0.006, "lookout_only": False,
            "starting_role": None}
    env = _vec(4, opts)
    assert env.generic_kernels
    env.close()
    _resume_equals_uninterrupted(tmp_path, 50, dict(game_options=opts), n_actions=6)


def test_resume_features_only(tmp_path):
    _resume_equals_uninterrupted(tmp_path, 200, dict(features=True, emit_grids=False))


def test_resume_without_auto_reset_past_done(tmp_path):
    _resume_equals_uninterrupted(tmp_path, 64, dict(game_options={"max_turns": 20, "chance_wolf_on_square": 0.01},
                                                    auto_reset=False, features=True))


@pytest.mark.parametrize("n", [1, 37, 1000])
def test_resume_ragged_batches(tmp_path, n):
    _resume_equals_uninterrupted(tmp_path, n, dict(features=True))


def test_resume_ego(tmp_path):
    _resume_equals_uninterrupted(tmp_path, 64, dict(game_options=OPTION_SETS["dense"][0], features=True), ego=True)


def test_reshard_one_handle_to_three():
    from wab_gym_b200.sharding import shard_range
    n = 1000
    acts = _acts(5, K1 + K2, n)
    kw = dict(game_options={"chance_wolf_on_square": 0.01}, features=True)
    a = _vec(n, seed=9, **kw)
    a.reset()
    _run(a, acts[:K1])
    sd = a.state_dict()
    tail = _run(a, acts[K1:])
    shards, parts = [], []
    for r in range(3):
        first, count = shard_range(n, r, 3)
        s = _vec(count, seed=9, env_id_base=first, **kw)
        s.reset()
        s.load_state_dict(sd)
        parts.append(_run(s, acts[K1:, first:first + count]))
        shards.append(s)
    joined = [{k: np.concatenate([p[t][k] for p in parts]) for k in tail[t]} for t in range(K2)]
    _same(tail, joined)
    totals = [s.stats() for s in shards]
    assert {k: sum(t[k] for t in totals) for k in totals[0]} == a.stats()
    st = [s.export_state() for s in shards]
    _same_state(a.export_state(), {k: np.concatenate([x[k] for x in st]) for k in st[0]})


def test_stale_centre_bush_is_reemitted():
    """A checkpoint right after a step that ate the bush under the ostrich empty: the loaded env shows that bush, exactly as
    the step's observation did, though its state has it gone."""
    opts = {"max_berries_per_bush": 1, "bush_power": 8, "turns_to_fill_food": 2, "chance_wolf_on_square": 0.004}
    n = 512
    env = _vec(n, opts, seed=4, features=True)
    obs = env.reset()
    rng = np.random.default_rng(1)
    for _ in range(60):
        on_bush = obs.grids[:, 1, 5, 5].cpu().numpy() == 1
        a = np.where(on_bush & (rng.random(n) < 0.8), 4, rng.integers(0, 5, n)).astype(np.uint8)
        obs, _, done, info = env.step(torch.from_numpy(a).cuda())
        ate = ((info["info"].cpu().numpy() >> 2) & 1).astype(bool) & ~done.cpu().numpy()
        st = env.export_state()
        gone = ((st["bush_mask"][:, 1] >> 28) & 1) == 0
        stale = np.nonzero(ate & gone & (obs.grids[:, 1, 5, 5].cpu().numpy() == 1))[0]
        if len(stale):
            break
    assert len(stale), "no env ate a bush empty"
    want = _host(obs, features=env.last_features)
    other = _vec(n, opts, seed=4, features=True)
    other.reset()
    got = _host(other.load_state_dict(env.state_dict()), features=other.last_features)
    for k in want:
        assert np.array_equal(got[k][stale], want[k][stale]), k
        assert np.array_equal(got[k], want[k]), k


def test_partial_load_changes_only_listed_slots():
    n = 64
    kw = dict(game_options={"chance_wolf_on_square": 0.01}, features=True)
    b, d = _vec(n, seed=2, **kw), _vec(n, seed=2, **kw)
    b.reset(); d.reset()
    acts = _acts(3, 30, n)
    last = _run(b, acts[:20])[-1]
    _run(d, acts)
    slots = [3, 10, 11, 40]
    before, donor = b.export_state(), d.export_state()
    got = _host(b.load_state(d.save_state(slots)), features=b.last_features)
    after = b.export_state()
    rest = np.setdiff1d(np.arange(n), slots)
    for k in before:
        assert np.array_equal(after[k][rest], before[k][rest]), k
        assert np.array_equal(after[k][slots], donor[k][slots]), k
    for k in got:
        assert np.array_equal(got[k][rest], last[k][rest]), k


@pytest.mark.parametrize("name", ["no_wolves", "defaults"])
def test_clone_shares_the_world(name):
    overrides = OPTION_SETS[name][0]
    n, i, j = 16, 2, 9
    env = _vec(n, overrides, seed=6, features=True)
    env.reset()
    acts = _acts(8, 15, n)
    _run(env, acts)
    obs = _host(env.load_state(env.save_state([j]), slots=[i]))
    for k in ("grids", "food", "role", "status"):
        assert np.array_equal(obs[k][i], obs[k][j]), k
    st = env.export_state()
    for k in ("x", "y", "food", "role", "status", "turn", "episode", "n_wolves", "wolves", "bush_mask", "n_log", "log"):
        assert np.array_equal(st[k][i], st[k][j]), k
    rng = np.random.default_rng(4)
    for t in range(200):
        a = torch.from_numpy(rng.integers(0, 5, n).astype(np.uint8))
        a[i] = a[j]
        o, _, done, _ = env.step(a.cuda())
        done = done.cpu().numpy()
        if done[i] or done[j]:
            break
        g = o.grids.cpu().numpy()
        if name == "no_wolves":
            for k, v in _host(o).items():
                assert np.array_equal(v[i], v[j]), (t, k)
        else:
            assert np.array_equal(g[i, 1], g[j, 1]), t          # bushes: the shared world; wolves: the slot's own draws
    else:
        pytest.fail("episode did not end")


def _guarded_out(env, G=256):
    raws = {}
    for k, v in list(env._out.items()):
        if v is None:
            continue
        nbytes = v.numel() * v.element_size()
        raw = torch.full((nbytes + 2 * G,), 0xAB, dtype=torch.uint8, device="cuda")
        raws[k] = raw
        env._out[k] = raw[G:G + nbytes].view(v.dtype).view(v.shape)
    return raws


def test_refused_loads_change_nothing():
    from wab_gym_b200 import _lib
    n, G = 40, 256
    kw = dict(game_options={"chance_wolf_on_square": 0.01}, features=True)
    src = _vec(n, seed=1, **kw)
    src.reset()
    _run(src, _acts(2, 25, n))
    sd = src.state_dict()
    for other in (dict(seed=2, **kw), dict(seed=1, game_options={"chance_wolf_on_square": 0.02}, features=True),
                  dict(seed=1, wolf_cap=32, **kw)):
        dst = _vec(n, **other)
        dst.reset()
        before = dst.export_state()
        with pytest.raises(ValueError):
            dst.load_state_dict(sd)
        _same_state(before, dst.export_state())
        dst.close()

    dst = _vec(n, seed=1, **kw)
    dst.reset()
    _run(dst, _acts(4, 5, n))
    raws = _guarded_out(dst)
    before = dst.export_state()
    good = src.save_state()
    for corrupt in ("n_wolves", "format"):
        rec = good.records.clone()
        if corrupt == "n_wolves":
            rec[7, 52:56] = torch.tensor([dst.game.wolf_cap + 1, 0, 0, 0], dtype=torch.uint8)
        else:
            rec[n - 1, 0] = 99
        with pytest.raises(ValueError, match="refused"):
            dst.load_state(good._replace(records=rec))
        _same_state(before, dst.export_state())
    with pytest.raises(ValueError):
        dst.load_state(good._replace(records=good.records[:1], env_ids=good.env_ids[:1]), slots=[n])
    # the device-side slot check on its own (the Python layer refuses such slots before calling)
    rejected = torch.zeros(1, dtype=torch.int32, device="cuda")
    bad_slots = torch.tensor([0, n], dtype=torch.int32, device="cuda")
    _lib.check(dst.lib.wab_vec_load_state(dst._h, ctypes.c_void_p(good.records.data_ptr()),
                                          ctypes.c_void_p(bad_slots.data_ptr()), 2, _lib.WabObs(0, 0, 0, 0),
                                          ctypes.c_void_p(rejected.data_ptr()), None))
    torch.cuda.synchronize()
    assert int(rejected.item()) == 1
    _same_state(before, dst.export_state())
    for k, raw in raws.items():
        assert int((raw[:G] != 0xAB).sum()) == 0 and int((raw[-G:] != 0xAB).sum()) == 0, k
    dst.load_state(good)                                   # and the untouched records do load
    _same_state(src.export_state(), dst.export_state())


def test_deepcopy_and_pickle_single_env():
    from wab_gym_b200.config import default_game_options
    from wab_gym_b200.env import WolvesAndBushesEnv
    env = WolvesAndBushesEnv(dict(default_game_options, chance_wolf_on_square=0.01), seed=3, env_id=5)
    rng = np.random.default_rng(0)
    for _ in range(17):
        env.step(int(rng.integers(0, 5)))
    for make in (copy.deepcopy, lambda e: pickle.loads(pickle.dumps(e))):
        dup = make(env)
        for x, y in zip(dup._get_obs(), env._get_obs()):
            assert np.array_equal(np.asarray(x), np.asarray(y))
        for a in rng.integers(0, 5, 100):
            o1, r1, d1, _ = env.step(int(a))
            o2, r2, d2, _ = dup.step(int(a))
            assert r1 == r2 and d1 == d2
            for x, y in zip(o1, o2):
                assert np.array_equal(np.asarray(x), np.asarray(y))
            if d1:
                env.reset(); dup.reset()
        dup.close()
        env.step(0)                                       # the original keeps working after the copy is gone
    env.close()


def test_rollout_resume_on_the_tcgen05_path_with_a_graph():
    from wab_gym_b200.policy import Policy, Rollout
    n = 1000
    torch.manual_seed(0)
    base = Policy(_vec(1, features=True).flat_dim, 5)

    def rollout(policy):
        env = _vec(n, seed=7, features=True)
        return Rollout(env, copy.deepcopy(policy), use_graph=True)

    def steps(ro, k):
        out = []
        for _ in range(k):
            ro.step()
            out.append((ro.actions.cpu().numpy().copy(), ro.values.cpu().numpy().copy(),
                        ro.env._out["reward"].cpu().numpy().copy()))
        return out

    a = rollout(base)
    assert a.tc_trunk and a.graph is not None
    steps(a, K1)
    want = steps(a, K2)
    b = rollout(base)
    steps(b, K1)
    sd = b.state_dict()
    c = rollout(Policy(b.env.flat_dim, 5))                # other weights, same shapes
    c.sample_seed ^= 1                                    # and another sampling seed: the graph is captured anew
    c.load_state_dict(sd)
    got = steps(c, K2)
    for t, (x, y) in enumerate(zip(want, got)):
        for u, v in zip(x, y):
            assert np.array_equal(u, v), t


@pytest.mark.parametrize("kernel", ["WAB2_GRID", "WAB2_NO_GRID"])
def test_world2_resume_and_reshard(monkeypatch, kernel):
    from wab_gym_b200.sharding import merge_state_dicts, shard_range
    from wab_gym_b200.world2 import VecWorld2
    monkeypatch.setenv(kernel, "1")
    n, dims = 96, (24, 24, 3, 2, 6)
    rng = np.random.default_rng(2)
    acts = [torch.from_numpy(np.concatenate([rng.integers(0, 6, (3, n)), rng.integers(0, 5, (2, n))]).astype(np.uint8)).cuda()
            for _ in range(K1 + K2)]

    def run(w, seq, reset_at=None):
        out = []
        for t, a in enumerate(seq):
            if t == reset_at:
                w.reset_environment()
            out.append([x.cpu().numpy().copy() for x in w.turn(a)])
        return out

    a = VecWorld2(n, *dims, seed=4)
    assert a.lib.wab2_kernel_kind(a._h) == (1 if kernel == "WAB2_GRID" else 0)
    run(a, acts[:K1], reset_at=10)
    halves = []
    for r in range(2):
        first, count = shard_range(n, r, 2)
        w = VecWorld2(count, *dims, seed=4, env_id_base=first)
        halves.append((first, count, w))
    sd = merge_state_dicts([a.state_dict()])
    want = run(a, acts[K1:], reset_at=30)
    b = VecWorld2(n, *dims, seed=4)
    b.load_state_dict(sd)
    got = run(b, acts[K1:], reset_at=30)
    for t, (x, y) in enumerate(zip(want, got)):
        for u, v in zip(x, y):
            assert np.array_equal(u, v), t
    parts = []
    for first, count, w in halves:
        w.load_state_dict(sd)
        parts.append(run(w, [x[:, first:first + count] for x in acts[K1:]], reset_at=30))
    for t in range(K2):
        for k in range(4):
            joined = np.concatenate([p[t][k] for p in parts], axis=1)
            assert np.array_equal(want[t][k], joined), (t, k)
    ea, eb = a.export_state(), b.export_state()
    assert np.array_equal(ea[0], eb[0]) and np.array_equal(ea[1], eb[1])
    other = VecWorld2(n, *dims, seed=5)
    with pytest.raises(ValueError, match="fingerprint"):
        other.load_state_dict(sd)
