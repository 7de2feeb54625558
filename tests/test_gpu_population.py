"""GPU tests of population self-play in one persistent launch (ocb_rollout_population_fused).

Slice s (128 worlds, both seats) plays weight set slice_policy[s] with its actor and critic.  Checked against the per-step
path (ocb_rollout_policy with the seat-major table slice_policy ++ slice_policy) bit for bit, against the single-policy
fused launch for a one-policy table, against the fp32 torch networks of each slice and the C oracle, through
PolicyRollout, across shards, and for its argument errors.
"""
import ctypes

import numpy as np
import pytest
import torch

from diverse_conventions_b200 import _native, layouts
from diverse_conventions_b200.overcooked_env import B200Overcooked, _ptr
from diverse_conventions_b200.policy import FusedPolicy, PolicyNet, log_softmax_sample
from diverse_conventions_b200.rollout import PolicyRollout, pair_tile_policy
from oracle.c_oracle import COracle

pytestmark = pytest.mark.gpu

ATOL_LOGP = 2e-4  # the tolerances of the suite's other policy tests
REL_TOL = 2e-4
N_POL = 8
OCB_ERR_INVALID_ARG = -1


def make_population(lp, n=N_POL, seed0=41):
    """n weight sets with distinct random weights; head gain 2, so sampled actions differ between policies"""
    actors = [PolicyNet("actor", lp.width, lp.height, lp.channels, 64).init_like_reference(seed0 + i, gain=2.0)
              for i in range(n)]
    critics = [PolicyNet("critic", lp.width, lp.height, lp.channels, 64).init_like_reference(seed0 + 500 + i)
               for i in range(n)]
    for net in actors + critics:
        for b in (net.conv_b, net.fc1_b, net.fc2_b, net.head_b):
            b.uniform_(-0.1, 0.1)
    pol = FusedPolicy(lp, 64, n)
    for i in range(n):
        pol.set_weights(i, actors[i], critics[i])
    return pol, actors, critics


def slice_table(kind, n_slices, n_pol=N_POL):
    """weight set per 128-world slice: 'distinct' (neighbours always differ; all distinct up to n_pol slices), 'runs'
    (runs of three equal slices), 'shuffled' (weight sets in a non-monotone, seeded random order)"""
    s = torch.arange(n_slices)
    if kind == "distinct":
        t = s % n_pol
    elif kind == "runs":
        t = (s // 3) % n_pol
    else:
        g = torch.Generator().manual_seed(n_slices)
        t = torch.randint(0, n_pol, (n_slices,), generator=g)
    return t.to(torch.int32)


def seat_major(table):
    return torch.cat([table, table])


def collect(env, pol, T, table, fused, seed, deterministic=False, rollouts=1, **kw):
    ro = PolicyRollout(env, pol, T, seat_major(table).to(env.sim_device), seed=seed, fused=fused, **kw)
    out = []
    for _ in range(rollouts):
        b = ro.collect(deterministic)
        torch.cuda.synchronize()
        out.append([x.clone() for x in (b.obs, b.actions, b.action_log_probs, b.value_preds, b.rewards, b.dones)])
    assert ro.fused == bool(fused)
    rs, ep = env.episode_stats()
    return out, env.get_state(), rs.clone(), ep.clone(), env.step_count


def assert_same(a, b):
    names = ("obs", "actions", "logp", "values", "rewards", "dones")
    for k in range(len(a[0])):
        for name, x, y in zip(names, a[0][k], b[0][k]):
            assert torch.equal(x, y), (k, name)
    assert np.array_equal(a[1], b[1])
    assert torch.equal(a[2], b[2]) and torch.equal(a[3], b[3]) and a[4] == b[4]


@pytest.mark.parametrize("deterministic", [0, 1])
@pytest.mark.parametrize("N,slots", [(1024, None), (8192, None), (32768, None), (32768, "1")])
@pytest.mark.parametrize("layout", ["simple", "random1", "unident_s", "random3"])
def test_population_launch_is_bit_identical_to_the_per_step_launches(monkeypatch, layout, N, slots, deterministic):
    """cramped_room (split mode at 8,192 worlds), coordination_ring, asymmetric_advantages (900-byte rows: no 16-byte
    loader), counter_circuit; 1,024 worlds (few CTAs), 8,192 (one round), 32,768 (two tiles in flight) and 32,768 with one
    tile in flight (several rounds per CTA, weights changing between rounds); three kinds of table each"""
    if slots is not None:
        monkeypatch.setenv("OCB_FUSED_SLOTS", slots)
    horizon, T = 9, 20  # several auto-resets inside one rollout
    lp = layouts.load_layout(layout, horizon)
    pol, _, _ = make_population(lp)
    for kind in ("distinct", "runs", "shuffled"):
        table = slice_table(kind, N // 128)
        res = []
        for fused in (False, True):
            env = B200Overcooked(layout, N, 0, horizon=horizon, seed=8)
            res.append(collect(env, pol, T, table, fused, seed=31, deterministic=bool(deterministic)))
            env.close()
        assert_same(res[0], res[1])
        assert res[1][4] == T


@pytest.mark.parametrize("layout,N", [("simple", 8192), ("random1", 32768)])
def test_one_policy_table_equals_the_single_policy_fused_launch(layout, N):
    """a table of one repeated weight set p fills the buffers of ocb_rollout_policy_fused(policy_index = p)"""
    horizon, T, p = 11, 24, 3
    lp = layouts.load_layout(layout, horizon)
    pol, _, _ = make_population(lp, 4)
    res = []
    for table in (None, torch.full((N // 128,), p, dtype=torch.int32)):
        env = B200Overcooked(layout, N, 0, horizon=horizon, seed=5)
        if table is None:
            ro = PolicyRollout(env, pol, T, seed=13, fused=True, policy_index=p)
            out = []
            for _ in range(2):
                b = ro.collect()
                torch.cuda.synchronize()
                out.append([x.clone() for x in (b.obs, b.actions, b.action_log_probs, b.value_preds, b.rewards, b.dones)])
            rs, ep = env.episode_stats()
            res.append((out, env.get_state(), rs.clone(), ep.clone(), env.step_count))
        else:
            res.append(collect(env, pol, T, table, True, seed=13, rollouts=2))
        env.close()
    assert_same(res[0], res[1])


@pytest.mark.parametrize("layout", ["simple", "random1"])
def test_each_slice_acts_with_its_own_networks_and_the_trajectory_replays_through_the_oracle(layout):
    horizon, T, wps = 15, 40, 256
    lp = layouts.load_layout(layout, horizon)
    pol, actors, critics = make_population(lp, 4)
    members = [2, 0, 3, 1]
    N = len(members) * wps
    table = pair_tile_policy([(m, m) for m in members], wps)
    env = B200Overcooked(layout, N, 0, horizon=horizon, seed=3)
    ro = PolicyRollout(env, pol, T, table.to(env.sim_device), seed=21)
    assert ro.fused is True
    buf = ro.collect()
    torch.cuda.synchronize()

    orc = COracle(lp, N)
    first = orc.observe()
    o, r, d = orc.rollout(buf.actions.cpu().numpy().astype(np.uint8))
    assert np.array_equal(buf.obs.cpu().numpy(), np.concatenate([first[None], o]))
    assert np.array_equal(buf.rewards.cpu().numpy(), r) and np.array_equal(buf.dones.cpu().numpy(), d)
    assert np.array_equal(env.get_state(), orc.state)
    assert d.sum() == N * (T // horizon)

    obs = buf.obs.cpu().reshape(T + 1, 2, len(members), wps, lp.width, lp.height, lp.channels)
    acts = buf.actions.cpu().reshape(T, 2, len(members), wps)
    logp = buf.action_log_probs.cpu().reshape(T, 2, len(members), wps)
    vals = buf.value_preds.cpu().reshape(T + 1, 2, len(members), wps)
    for k, m in enumerate(members):
        for t in (0, T // 2, T - 1, T):
            rows = obs[t, :, k].reshape(-1, lp.width, lp.height, lp.channels)
            ref_v = critics[m].forward(rows)[:, 0]
            assert float((vals[t, :, k].reshape(-1) - ref_v).abs().max() / ref_v.abs().max()) < REL_TOL, (k, t)
            if t < T:
                ref_lp = log_softmax_sample(actors[m].forward(rows), acts[t, :, k].reshape(-1))
                assert torch.allclose(logp[t, :, k].reshape(-1), ref_lp, atol=ATOL_LOGP), (k, t)

    # per-member scores: the device's per-slice read-out equals the oracle's episode returns
    rs, ep = ro.slice_episode_returns(wps)
    ret, total = np.zeros(N, dtype=np.int64), np.zeros(N, dtype=np.int64)
    for t in range(T):
        ret += r[t, 0]
        total[d[t] != 0] += ret[d[t] != 0]
        ret[d[t] != 0] = 0
    assert np.array_equal(rs.cpu().numpy(), total.reshape(len(members), wps).sum(1))
    assert np.array_equal(ep.cpu().numpy(), d.reshape(T, len(members), wps).sum((0, 2)))
    env.close()


def test_policy_rollout_picks_the_population_launch_and_matches_per_step_under_graph_replays():
    layout, horizon, T, wps = "random1", 13, 30, 512
    lp = layouts.load_layout(layout, horizon)
    pol, _, _ = make_population(lp, 4)
    table = pair_tile_policy([(1, 1), (3, 3), (0, 0), (2, 2)], wps)
    N = 4 * wps
    res = []
    for use_graph in (False, True):
        for fused in (None, False):
            env = B200Overcooked(layout, N, 0, horizon=horizon, seed=6)
            ro = PolicyRollout(env, pol, T, table.to(env.sim_device), seed=4, fused=fused, use_graph=use_graph)
            assert ro.fused is (fused is None)
            out = []
            for _ in range(3):  # replays of a captured graph draw fresh actions from the device step counter
                b = ro.collect()
                torch.cuda.synchronize()
                out.append([x.clone() for x in (b.obs, b.actions, b.action_log_probs, b.value_preds, b.rewards, b.dones)])
            assert ro.fused is (fused is None)
            rs, ep = env.episode_stats()
            res.append((out, env.get_state(), rs.clone(), ep.clone(), env.step_count))
            env.close()
    for other in res[1:]:
        assert_same(res[0], other)
    assert not torch.equal(res[0][0][0][1], res[0][0][1][1])


def test_mixed_table_with_a_critic_stays_on_per_step_launches():
    lp = layouts.load_layout("simple", 400)
    pol, _, _ = make_population(lp, 2)
    env = B200Overcooked("simple", 256, 0, horizon=400, seed=1)
    ro = PolicyRollout(env, pol, 5, pair_tile_policy([(0, 1), (1, 0)], 128, env.sim_device))
    assert ro.fused is False
    ro.collect()
    torch.cuda.synchronize()
    assert ro.fused is False
    with pytest.raises(ValueError):
        PolicyRollout(env, pol, 5, pair_tile_policy([(0, 1), (1, 0)], 128, env.sim_device), fused=True)
    env.close()


@pytest.mark.parametrize("layout,hidden", [("simple", 512), ("schelling", 64)])
def test_fused_true_raises_where_the_population_launch_does_not_apply(layout, hidden):
    """hidden 512 and a generic-kernel layout (9-row grid): OCB_ERR_UNSUPPORTED -> NativeError; fused=None falls back"""
    lp = layouts.load_layout(layout, 400)
    pol = FusedPolicy(lp, hidden, 2)
    for i in range(2):
        pol.set_weights(i, PolicyNet("actor", lp.width, lp.height, lp.channels, hidden).init_like_reference(i),
                        PolicyNet("critic", lp.width, lp.height, lp.channels, hidden).init_like_reference(50 + i))
    env = B200Overcooked(layout, 256, 0, horizon=400, seed=1)
    table = pair_tile_policy([(0, 0), (1, 1)], 128, env.sim_device)
    with pytest.raises(_native.NativeError) as e:
        PolicyRollout(env, pol, 3, table, fused=True).collect()
    assert e.value.code == _native.OCB_ERR_UNSUPPORTED
    ro = PolicyRollout(env, pol, 3, table)
    ro.collect()
    torch.cuda.synchronize()
    assert ro.fused is False
    env.close()


@pytest.mark.parametrize("layout", ["simple", "random1"])
def test_sharded_population_reproduces_the_whole(layout):
    """two env handles of half the worlds each, sampling keyed by the global (seat, world), fill the whole run's buffers"""
    horizon, T, N = 17, 25, 4096
    lp = layouts.load_layout(layout, horizon)
    pol, _, _ = make_population(lp)
    table = slice_table("shuffled", N // 128)
    env = B200Overcooked(layout, N, 0, horizon=horizon, seed=9)
    whole = collect(env, pol, T, table, True, seed=2, total_worlds=N)
    env.close()
    h = N // 2
    for part in range(2):
        off = part * h
        env = B200Overcooked(layout, h, 0, horizon=horizon, seed=9, world_offset=off)
        got = collect(env, pol, T, table[off // 128:(off + h) // 128], True, seed=2, world_offset=off, total_worlds=N)
        env.close()
        for name, x, y in zip(("obs", "actions", "logp", "values", "rewards"), whole[0][0][:5], got[0][0][:5]):
            assert torch.equal(x[:, :, off:off + h], y), name
        assert torch.equal(whole[0][0][5][:, off:off + h], got[0][0][5])
        assert torch.equal(whole[2][off:off + h], got[2]) and torch.equal(whole[3][off:off + h], got[3])


def test_argument_errors_launch_nothing():
    lp = layouts.load_layout("simple", 400)
    pol, _, _ = make_population(lp, 2)
    lib = _native.lib()
    for N, with_values in ((256, False), (192, True)):
        env = B200Overcooked("simple", N, 0, horizon=400, seed=1)
        dev = env.sim_device
        table = torch.zeros((N + 127) // 128, dtype=torch.int32, device=dev)
        obs = torch.zeros((5, 2, N, lp.width, lp.height, lp.channels), dtype=torch.int8, device=dev)
        actions = torch.full((4, 2, N), -7, dtype=torch.int32, device=dev)
        values = torch.zeros((5, 2, N), dtype=torch.float32, device=dev) if with_values else None
        state = env.get_state()
        stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        rc = lib.ocb_rollout_population_fused(env._h, pol._h, 4, _ptr(table), _ptr(obs), _ptr(actions), None, _ptr(values),
                                              None, None, 0, 1, stream)
        torch.cuda.synchronize()
        assert rc == OCB_ERR_INVALID_ARG
        assert (actions == -7).all() and int(obs.abs().sum()) == 0
        assert np.array_equal(env.get_state(), state) and env.step_count == 0
        env.close()
