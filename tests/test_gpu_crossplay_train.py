"""Cross-play training rollouts on the device (ocb_rollout_crossplay_train_fused): the cross-play launch, then one critic pass
that values each 128-row seat tile with the critic its critic_policy entry names, or not at all for -1.

Checked against the per-step path (PolicyRollout(tile_policy, with_critic=True, fused=False)) bit for bit, against
FusedPolicy.value and the fp32 torch critics for critic sets that differ from the actor sets, against the cross-play launch
for the trajectory, under graph replay and sharding, on the fallback, and for its argument errors.  The CPU test at the end
covers crossplay_training_tables.
"""
import ctypes

import numpy as np
import pytest
import torch

from diverse_conventions_b200 import _native, layouts
from diverse_conventions_b200.rollout import crossplay_training_tables, pair_tile_policy

OCB_ERR_INVALID_ARG = -1
REL_TOL = 2e-4  # the suite's tolerance of the tensor-core networks against fp32
SENTINEL = 12345.0


def make_population(lp, n, hidden=64, seed0=41):
    """n weight sets with distinct random weights; head gain 2, so sampled actions differ between policies"""
    from diverse_conventions_b200.policy import FusedPolicy, PolicyNet
    actors = [PolicyNet("actor", lp.width, lp.height, lp.channels, hidden).init_like_reference(seed0 + i, gain=2.0)
              for i in range(n)]
    critics = [PolicyNet("critic", lp.width, lp.height, lp.channels, hidden).init_like_reference(seed0 + 500 + i)
               for i in range(n)]
    for net in actors + critics:
        for b in (net.conv_b, net.fc1_b, net.fc2_b, net.head_b):
            b.uniform_(-0.1, 0.1)
    pol = FusedPolicy(lp, hidden, n)
    for i in range(n):
        pol.set_weights(i, actors[i], critics[i])
    return pol, actors, critics


def mixed_table(n_tiles, n_pol, seed):
    """an actor table that gives the two seats different policies on most tiles"""
    g = torch.Generator().manual_seed(seed)
    return torch.randint(0, n_pol, (n_tiles,), generator=g).to(torch.int32)


def collect(env, pol, T, table, seed, fused, critic=None, deterministic=False, rollouts=1, **kw):
    from diverse_conventions_b200.rollout import PolicyRollout
    dev = env.sim_device
    ro = PolicyRollout(env, pol, T, table.to(dev), seed=seed, fused=fused,
                       critic_policy=None if critic is None else critic.to(dev), **kw)
    out = []
    for _ in range(rollouts):
        b = ro.collect(deterministic)
        torch.cuda.synchronize()
        out.append([None if x is None else x.clone()
                    for x in (b.obs, b.actions, b.action_log_probs, b.value_preds, b.rewards, b.dones)])
    rs, ep = env.episode_stats()
    return out, env.get_state(), rs.clone(), ep.clone(), env.step_count, ro.fused


def assert_same(a, b, skip_values=False):
    names = ("obs", "actions", "logp", "values", "rewards", "dones")
    for k in range(len(a[0])):
        for name, x, y in zip(names, a[0][k], b[0][k]):
            if not (skip_values and name == "values"):
                assert torch.equal(x, y), (k, name)
    assert np.array_equal(a[1], b[1])
    assert torch.equal(a[2], b[2]) and torch.equal(a[3], b[3]) and a[4] == b[4]


def tile_values(values, T, n_tiles):
    return values.view(T + 1, n_tiles, 128)


@pytest.mark.gpu
@pytest.mark.parametrize("deterministic", [0, 1])
@pytest.mark.parametrize("N", [1024, 32768])
@pytest.mark.parametrize("layout", ["simple", "random1", "random3", "unident_s"])
def test_equals_the_per_step_path_when_every_tile_is_valued_by_its_actor_set(layout, N, deterministic):
    """critic_policy == tile_policy: every buffer, the final env state, the episode statistics and the step counter equal
    PolicyRollout(tile_policy, with_critic=True, fused=False), over two consecutive collections with auto-resets inside T;
    1,024 worlds (16 seat tiles) and 32,768 (two world tiles in flight per SM)"""
    from diverse_conventions_b200.overcooked_env import B200Overcooked
    horizon, T, n_pol = 9, 20, 6
    lp = layouts.load_layout(layout, horizon)
    pol, _, _ = make_population(lp, n_pol)
    table = mixed_table(2 * N // 128, n_pol, N + len(layout))
    res = []
    for fused in (False, None):
        env = B200Overcooked(layout, N, 0, horizon=horizon, seed=8)
        res.append(collect(env, pol, T, table, 31, fused, critic=None if fused is False else table,
                           deterministic=bool(deterministic), rollouts=2))
        env.close()
    assert res[0][5] is False and res[1][5] is True
    assert_same(res[0], res[1])
    assert res[1][4] == 2 * T


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["simple", "unident_s"])
def test_tiles_without_a_critic_are_never_written(layout):
    """critic_policy with -1 entries clustered (a whole seat half), scattered, everywhere and nowhere: the other tiles' values
    equal the per-step path's; through the C entry point the -1 slots keep a sentinel, through PolicyRollout they are 0.0"""
    from diverse_conventions_b200.overcooked_env import B200Overcooked, _ptr
    horizon, T, N, n_pol = 9, 15, 2048, 4
    n_tiles = 2 * N // 128
    lp = layouts.load_layout(layout, horizon)
    pol, _, _ = make_population(lp, n_pol)
    table = mixed_table(n_tiles, n_pol, 3)
    env = B200Overcooked(layout, N, 0, horizon=horizon, seed=2)
    ref = collect(env, pol, T, table, 5, False, rollouts=2)
    env.close()
    ref_v = [tile_values(ref[0][k][3], T, n_tiles).cpu() for k in range(2)]
    g = torch.Generator().manual_seed(7)
    scattered = table.clone()
    scattered[torch.rand(n_tiles, generator=g) < 0.5] = -1
    clustered = table.clone()
    clustered[n_tiles // 2:] = -1
    lib = _native.lib()
    for name, critic in (("clustered", clustered), ("scattered", scattered), ("everywhere", torch.full_like(table, -1)),
                         ("nowhere", table)):
        none = critic < 0
        # the C entry point: slots of -1 tiles keep what was there
        env = B200Overcooked(layout, N, 0, horizon=horizon, seed=2)
        dev = env.sim_device
        obs = torch.empty((T + 1, 2, N, lp.width, lp.height, lp.channels), dtype=torch.int8, device=dev)
        actions = torch.empty((T, 2, N), dtype=torch.int32, device=dev)
        values = torch.full((T + 1, 2, N), SENTINEL, dtype=torch.float32, device=dev)
        t_dev, c_dev = table.to(dev), critic.to(dev)
        _native.check(lib.ocb_observe(env._h, _ptr(obs[0]), env._stream()))
        stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        _native.check(lib.ocb_rollout_crossplay_train_fused(env._h, pol._h, T, _ptr(t_dev), _ptr(c_dev), _ptr(obs),
                                                            _ptr(actions), None, _ptr(values), None, None, 0, 5, stream))
        torch.cuda.synchronize()
        env.close()
        v = tile_values(values, T, n_tiles).cpu()
        assert torch.equal(obs, ref[0][0][0]) and torch.equal(actions, ref[0][0][1]), name
        assert (v[:, none] == SENTINEL).all(), name
        assert torch.equal(v[:, ~none], ref_v[0][:, ~none]), name
        # PolicyRollout: the buffer is zero-initialised and -1 slots stay 0.0
        env = B200Overcooked(layout, N, 0, horizon=horizon, seed=2)
        got = collect(env, pol, T, table, 5, None, critic=critic, rollouts=2)
        env.close()
        assert got[5] is True
        for k in range(2):
            v = tile_values(got[0][k][3], T, n_tiles).cpu()
            assert (v[:, none] == 0.0).all(), name
            assert torch.equal(v[:, ~none], ref_v[k][:, ~none]), name
        assert_same(ref, got, skip_values=True)


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["simple", "random1"])
def test_xd_critics_that_differ_from_the_actors(layout):
    """XD's layout: ego 0 with its SP critic (set 1) on an SP slice, XP critics (sets 4 / 5 seat 0, 6 / 7 seat 1) against
    partners 2 and 3 (no critic).  Values equal FusedPolicy.value on the recorded observations with the critic table, bit for
    bit, and the fp32 torch critics at 2e-4; the trajectory equals ocb_rollout_crossplay_fused's with the same seed"""
    from diverse_conventions_b200.overcooked_env import B200Overcooked
    horizon, T, wps = 13, 24, 256
    lp = layouts.load_layout(layout, horizon)
    pol, actors, critics = make_population(lp, 8)
    partners, xp0, xp1 = [2, 3], [4, 5], [6, 7]
    slices = ([((0, 1), (0, 1))] + [((0, xp0[j]), (p, None)) for j, p in enumerate(partners)] +
              [((p, None), (0, xp1[j])) for j, p in enumerate(partners)])
    tile, critic = crossplay_training_tables(slices, wps)
    N = len(slices) * wps
    n_tiles = 2 * N // 128
    env = B200Overcooked(layout, N, 0, horizon=horizon, seed=3)
    got = collect(env, pol, T, tile, 9, None, critic=critic)
    env.close()
    assert got[5] is True
    env = B200Overcooked(layout, N, 0, horizon=horizon, seed=3)
    xp = collect(env, pol, T, tile, 9, True, with_critic=False)
    env.close()
    for name, i in (("obs", 0), ("actions", 1), ("logp", 2), ("rewards", 4), ("dones", 5)):
        assert torch.equal(got[0][0][i], xp[0][0][i]), name
    assert np.array_equal(got[1], xp[1]) and got[4] == xp[4]

    obs, values = got[0][0][0], got[0][0][3]
    dev = obs.device
    filled = critic.clamp(min=0).to(dev)
    has = (critic >= 0).to(dev)
    for t in range(T + 1):
        v = pol.value(obs[t], tile_policy=filled).view(n_tiles, 128)
        assert torch.equal(values[t].view(n_tiles, 128)[has], v[has]), t
        assert (values[t].view(n_tiles, 128)[~has] == 0.0).all(), t
    rows = obs.view(T + 1, 2, N, lp.width, lp.height, lp.channels)
    for t in (0, T // 2, T):
        for s, sl in enumerate(slices):
            for seat in range(2):
                c = sl[seat][1]
                if c is None:
                    continue
                x = rows[t, seat, s * wps:(s + 1) * wps].cpu()
                ref = critics[c].forward(x)[:, 0]
                v = values[t, seat, s * wps:(s + 1) * wps].cpu()
                assert float((v - ref).abs().max() / ref.abs().max()) < REL_TOL, (t, s, seat)


@pytest.mark.gpu
def test_graph_replay_equals_eager_issue_and_shards_reproduce_the_whole():
    from diverse_conventions_b200.overcooked_env import B200Overcooked
    layout, horizon, T, wps = "random1", 11, 18, 512
    lp = layouts.load_layout(layout, horizon)
    pol, _, _ = make_population(lp, 5)
    slices = [((0, 0), (0, 0)), ((0, 4), (1, None)), ((2, None), (0, 3)), ((0, 0), (3, None))]
    tile, critic = crossplay_training_tables(slices, wps)
    N = len(slices) * wps
    res = []
    for use_graph in (False, True):
        env = B200Overcooked(layout, N, 0, horizon=horizon, seed=6)
        res.append(collect(env, pol, T, tile, 4, None, critic=critic, rollouts=3, use_graph=use_graph))
        env.close()
    assert res[0][5] is True and res[1][5] is True
    assert_same(res[0], res[1])
    assert not torch.equal(res[0][0][0][1], res[0][0][1][1])  # replays draw fresh actions

    env = B200Overcooked(layout, N, 0, horizon=horizon, seed=9)
    whole = collect(env, pol, T, tile, 2, None, critic=critic, total_worlds=N)
    env.close()
    h, half = N // 2, tile.numel() // 2
    for part in range(2):
        off = part * h
        sl = lambda t: torch.cat([t[off // 128:(off + h) // 128], t[half + off // 128:half + (off + h) // 128]])
        env = B200Overcooked(layout, h, 0, horizon=horizon, seed=9, world_offset=off)
        got = collect(env, pol, T, sl(tile), 2, None, critic=sl(critic), world_offset=off, total_worlds=N)
        env.close()
        for name, x, y in zip(("obs", "actions", "logp", "values", "rewards"), whole[0][0][:5], got[0][0][:5]):
            assert torch.equal(x[:, :, off:off + h], y), name
        assert torch.equal(whole[0][0][5][:, off:off + h], got[0][0][5])
        assert torch.equal(whole[2][off:off + h], got[2]) and torch.equal(whole[3][off:off + h], got[3])


@pytest.mark.gpu
@pytest.mark.parametrize("layout,hidden", [("simple", 512), ("schelling", 64)])
def test_fallback_where_the_fused_path_is_unsupported(layout, hidden):
    """hidden 512 and a generic-kernel layout: fused=None falls back to per-step launches with the same semantics (values of
    the named critics against torch, -1 slots 0.0, also after a graph replay); fused=True raises OCB_ERR_UNSUPPORTED"""
    from diverse_conventions_b200.overcooked_env import B200Overcooked
    from diverse_conventions_b200.rollout import PolicyRollout
    horizon, T, wps = 7, 9, 128
    lp = layouts.load_layout(layout, horizon)
    pol, _, critics = make_population(lp, 3, hidden=hidden)
    slices = [((0, 1), (2, None)), ((2, None), (0, 0))]
    tile, critic = crossplay_training_tables(slices, wps)
    N = len(slices) * wps
    env = B200Overcooked(layout, N, 0, horizon=horizon, seed=1)
    dev = env.sim_device
    with pytest.raises(_native.NativeError) as e:
        PolicyRollout(env, pol, T, tile.to(dev), fused=True, critic_policy=critic.to(dev)).collect()
    assert e.value.code == _native.OCB_ERR_UNSUPPORTED
    for use_graph in (False, True):
        ro = PolicyRollout(env, pol, T, tile.to(dev), critic_policy=critic.to(dev), use_graph=use_graph)
        for _ in range(2):
            b = ro.collect()
            torch.cuda.synchronize()
        assert ro.fused is False
        rows = b.obs.view(T + 1, 2, N, -1)
        for t in (0, T):
            for s, sl in enumerate(slices):
                for seat in range(2):
                    v = b.value_preds[t, seat, s * wps:(s + 1) * wps].cpu()
                    c = sl[seat][1]
                    if c is None:
                        assert (v == 0.0).all()
                        continue
                    x = rows[t, seat, s * wps:(s + 1) * wps].cpu().view(wps, lp.width, lp.height, lp.channels)
                    ref = critics[c].forward(x)[:, 0]
                    assert float((v - ref).abs().max() / ref.abs().max()) < REL_TOL, (t, s, seat)
    ro = PolicyRollout(env, pol, T, tile.to(dev), critic_policy=critic.to(dev), fused=False)
    ro.collect()
    torch.cuda.synchronize()
    assert ro.fused is False
    env.close()


@pytest.mark.gpu
def test_argument_errors():
    from diverse_conventions_b200.overcooked_env import B200Overcooked, _ptr
    from diverse_conventions_b200.rollout import PolicyRollout
    lp = layouts.load_layout("simple", 400)
    pol, _, _ = make_population(lp, 2)
    lib = _native.lib()

    def call(env, pol_h, T, tile, critic, obs, actions, values):
        stream = ctypes.c_void_p(torch.cuda.current_stream(env.sim_device).cuda_stream)
        rc = lib.ocb_rollout_crossplay_train_fused(env._h, pol_h, T, _ptr(tile), _ptr(critic), obs, _ptr(actions), None,
                                                   _ptr(values), None, None, 0, 1, stream)
        torch.cuda.synchronize()
        return rc, lib.ocb_last_error().decode()

    for N in (256, 192):
        env = B200Overcooked("simple", N, 0, horizon=400, seed=1)
        dev = env.sim_device
        n_tiles = (2 * N + 127) // 128
        tile = torch.zeros(n_tiles, dtype=torch.int32, device=dev)
        obs = torch.zeros((6, 2, N, lp.width, lp.height, lp.channels), dtype=torch.int8, device=dev)
        actions = torch.full((5, 2, N), -7, dtype=torch.int32, device=dev)
        values = torch.full((6, 2, N), SENTINEL, dtype=torch.float32, device=dev)
        state = env.get_state()
        cases = [(tile, tile, _ptr(obs), actions, None, OCB_ERR_INVALID_ARG, "required"),
                 (tile, None, _ptr(obs), actions, values, OCB_ERR_INVALID_ARG, "critic_policy"),
                 (None, tile, _ptr(obs), actions, values, OCB_ERR_INVALID_ARG, "tile_policy"),
                 (tile, tile, None, actions, values, OCB_ERR_INVALID_ARG, "required"),
                 (tile, tile, ctypes.c_void_p(obs.data_ptr() + 2), actions, values, OCB_ERR_INVALID_ARG, "aligned")]
        if N % 128:
            cases.append((tile, tile, _ptr(obs), actions, values, OCB_ERR_INVALID_ARG, "multiple of 128"))
        for t_, c_, o_, a_, v_, code, msg in cases:
            rc, err = call(env, pol._h, 5, t_, c_, o_, a_, v_)
            assert rc == code and msg in err, (N, msg, rc, err)
        assert (actions == -7).all() and int(obs.abs().sum()) == 0 and (values == SENTINEL).all()
        assert np.array_equal(env.get_state(), state) and env.step_count == 0
        env.close()

    env = B200Overcooked("simple", 256, 0, horizon=400, seed=1)
    dev = env.sim_device
    pol512 = make_population(lp, 1, hidden=512)[0]
    tile = torch.zeros(4, dtype=torch.int32, device=dev)
    obs = torch.zeros((6, 2, 256, lp.width, lp.height, lp.channels), dtype=torch.int8, device=dev)
    actions = torch.full((5, 2, 256), -7, dtype=torch.int32, device=dev)
    values = torch.full((6, 2, 256), SENTINEL, dtype=torch.float32, device=dev)
    rc, err = call(env, pol512._h, 5, tile, tile, _ptr(obs), actions, values)
    assert rc == _native.OCB_ERR_UNSUPPORTED and "hidden_size 64" in err
    assert (actions == -7).all() and (values == SENTINEL).all() and env.step_count == 0

    # Python: critic_policy needs tile_policy and the critic, the table shape, entries in range, whole seat tiles
    t = pair_tile_policy([(0, 1), (1, 0)], 128, dev)
    bad = [dict(tile_policy=None, critic_policy=t), dict(tile_policy=t, critic_policy=t, with_critic=False),
           dict(tile_policy=t, critic_policy=t.to(torch.int64)), dict(tile_policy=t, critic_policy=t[:2]),
           dict(tile_policy=t, critic_policy=torch.tensor([0, 2, 1, 0], dtype=torch.int32, device=dev)),
           dict(tile_policy=t, critic_policy=torch.tensor([0, -2, 1, 0], dtype=torch.int32, device=dev)),
           dict(tile_policy=torch.tensor([0, -1, 1, 0], dtype=torch.int32, device=dev), critic_policy=t)]
    for kw in bad:
        with pytest.raises(ValueError):
            PolicyRollout(env, pol, 5, **kw)
    env.close()
    env = B200Overcooked("simple", 192, 0, horizon=400, seed=1)
    t3 = torch.zeros(3, dtype=torch.int32, device=env.sim_device)
    with pytest.raises(ValueError):
        PolicyRollout(env, pol, 5, t3, critic_policy=t3)
    env.close()


def test_crossplay_training_tables_for_xd_and_best_response():
    """CPU: seat-major tables, 128-world tiles, None -> -1"""
    xd = [((0, 1), (0, 1)), ((0, 4), (2, None)), ((0, 5), (3, None)), ((2, None), (0, 6)), ((3, None), (0, 7))]
    tile, critic = crossplay_training_tables(xd, 256)
    rep = lambda v: [x for x in v for _ in range(2)]
    assert tile.dtype == torch.int32 and critic.dtype == torch.int32
    assert tile.tolist() == rep([0, 0, 0, 2, 3]) + rep([0, 2, 3, 0, 0])
    assert critic.tolist() == rep([1, 4, 5, -1, -1]) + rep([1, -1, -1, 6, 7])
    br = [((0, 0), (p, None)) for p in (1, 2, 3, 4)] + [((p, None), (0, 0)) for p in (1, 2, 3, 4)]
    tile, critic = crossplay_training_tables(br, 128)
    assert tile.tolist() == [0, 0, 0, 0, 1, 2, 3, 4] + [1, 2, 3, 4, 0, 0, 0, 0]
    assert critic.tolist() == [0, 0, 0, 0, -1, -1, -1, -1] + [-1, -1, -1, -1, 0, 0, 0, 0]
    assert torch.equal(tile, pair_tile_policy([(s[0][0], s[1][0]) for s in br], 128))
    with pytest.raises(ValueError):
        crossplay_training_tables(xd, 100)
    with pytest.raises(ValueError):
        crossplay_training_tables([((0, 1),)], 128)
