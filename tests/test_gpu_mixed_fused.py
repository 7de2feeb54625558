"""GPU tests of the mixed-play collection in one persistent launch (ocb_rollout_mixed_fused).

The fused collection is checked bit for bit against the per-step collection (ocb_rollout_mixed) run on an identical env:
every buffer, the final env state, the step counter and the episode statistics.  Shapes cover ragged last tiles, tiles
filled exactly, two tiles in flight per CTA (more than 148 x 64 worlds), episodes ending inside the collection, sampled and
greedy actions, other weight-set pairs, the actor-only variant and consecutive collections.  Both paths are also checked
against the step-by-step reconstruction of test_gpu_mixed, and the collector's graph replay, fallback and argument errors.
"""
import ctypes

import numpy as np
import pytest
import torch

from diverse_conventions_b200 import _native, layouts
from diverse_conventions_b200.mixed import MixedPlayBuffer, MixedPlayCollector
from diverse_conventions_b200.overcooked_env import B200Overcooked, _ptr
from diverse_conventions_b200.policy import FusedPolicy, PolicyNet
from oracle import mixed_oracle as mo
from test_gpu_mixed import reconstruct
from test_gpu_rollout import make_policies

pytestmark = pytest.mark.gpu

OCB_ERR_INVALID_ARG = -1
NAMES = ("obs", "actions", "logp", "values", "rewards", "dones")


def run(layout, pol, L, replicas, fused, horizon=7, main=0, partner=1, deterministic=0, critic=True, collections=1,
        seed=77, mix_seed=4242):
    """collections through the C entry points on a fresh env advanced by a random prefix -> buffers per collection,
    final state, episode statistics, step count"""
    N = replicas * (L - 1)
    env = B200Overcooked(layout, N, 0, horizon=horizon, seed=5)
    env.rollout_random(3)
    lib = _native.lib()
    dev = env.sim_device
    scratch = None if fused else torch.empty((int(lib.ocb_rollout_mixed_scratch_bytes(env._h)),), dtype=torch.uint8,
                                             device=dev)
    buf = MixedPlayBuffer(env, L)
    out = []
    for c in range(collections):
        for t in (buf.obs, buf.actions, buf.action_log_probs, buf.value_preds, buf.rewards, buf.dones):
            t.fill_(-7)  # cells neither path writes keep it
        stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        args = (env._h, pol._h, L, main, partner, _ptr(buf.obs), _ptr(buf.actions),
                _ptr(buf.action_log_probs) if critic else None, _ptr(buf.value_preds) if critic else None,
                _ptr(buf.rewards), _ptr(buf.dones), deterministic, seed + c, mix_seed + c)
        if fused:
            _native.check(lib.ocb_rollout_mixed_fused(*args, stream))
        else:
            _native.check(lib.ocb_rollout_mixed(*args, _ptr(scratch), scratch.numel(), stream))
        torch.cuda.synchronize()
        out.append([t.clone() for t in (buf.obs, buf.actions, buf.action_log_probs, buf.value_preds, buf.rewards,
                                        buf.dones)])
    rs, ep = env.episode_stats()
    torch.cuda.synchronize()
    res = (out, env.get_state(), rs.clone(), ep.clone(), env.step_count)
    env.close()
    return res


def assert_same(a, b):
    for k in range(len(a[0])):
        for name, x, y in zip(NAMES, a[0][k], b[0][k]):
            assert torch.equal(x, y), (k, name)
    assert np.array_equal(a[1], b[1])
    assert torch.equal(a[2], b[2]) and torch.equal(a[3], b[3]) and a[4] == b[4]


@pytest.fixture(scope="module")
def policies():
    cache = {}

    def get(layout):
        if layout not in cache:
            cache[layout] = make_policies(layouts.load_layout(layout, 7), 2)[0]
        return cache[layout]
    return get


@pytest.mark.parametrize("deterministic", [0, 1])
@pytest.mark.parametrize("L,replicas", [(9, 5), (6, 27), (9, 64), (5, 2400)])
@pytest.mark.parametrize("layout", ["simple", "random1", "unident_s", "random3"])
def test_fused_collection_is_bit_identical_to_the_per_step_collection(policies, layout, L, replicas, deterministic):
    """40 and 135 worlds (ragged last tile), 512 (64-world tiles filled exactly), 9,600 (more tiles than SMs: two tiles
    in flight where the layout's planes fit twice); horizon 7, so episodes end inside the collection"""
    pol = policies(layout)
    per_step = run(layout, pol, L, replicas, False, deterministic=deterministic)
    fused = run(layout, pol, L, replicas, True, deterministic=deterministic)
    assert_same(per_step, fused)
    assert fused[4] == 3 + 2 * L
    assert int(fused[0][0][5].sum()) > 0  # an episode ended inside the collection


@pytest.mark.parametrize("variant", ["main1", "same", "actor_only", "two_collections"])
@pytest.mark.parametrize("layout", ["simple", "random1"])
def test_fused_collection_variants(policies, layout, variant):
    """main_policy != 0, main == partner, no critic and no log-probs, and a second collection continuing the first"""
    pol = policies(layout)
    kw = {"main1": dict(main=1, partner=0), "same": dict(main=1, partner=1), "actor_only": dict(critic=False),
          "two_collections": dict(collections=2)}[variant]
    per_step = run(layout, pol, 7, 20, False, **kw)
    fused = run(layout, pol, 7, 20, True, **kw)
    assert_same(per_step, fused)
    if variant == "actor_only":
        assert bool((fused[0][0][3] == -7).all()) and bool((fused[0][0][2] == -7).all())


@pytest.mark.parametrize("fused", [True, False])
@pytest.mark.parametrize("layout,L,replicas", [("simple", 9, 5), ("random1", 6, 27), ("unident_s", 8, 10),
                                               ("random3", 7, 12)])
def test_both_paths_match_the_stepwise_reconstruction(layout, L, replicas, fused):
    horizon = 7
    N = replicas * (L - 1)
    lp = layouts.load_layout(layout, horizon)
    pol, _, _ = make_policies(lp, 2)
    env = B200Overcooked(layout, N, 0, horizon=horizon, seed=5)
    env.rollout_random(3)
    torch.cuda.synchronize()
    state0, step0 = env.get_state().copy(), env.step_count
    seed, mix_seed = 77, 4242
    col = MixedPlayCollector(env, pol, L, 0, 1, seed=seed, mix_seed=mix_seed, fused=fused)
    buf = col.collect()
    torch.cuda.synchronize()
    assert col.fused is fused
    assert env.step_count == step0 + 2 * L

    st, use, orc = reconstruct(lp, pol, L, N, seed, mix_seed, step0, state0)
    assert np.array_equal(env.get_state(), orc.state)
    assert (st["played"] != st["actions"]).any()
    assert np.array_equal(buf.obs[:L].cpu().numpy(), mo.place(L, st["obs"], world_axis=1))
    assert np.array_equal(buf.actions.cpu().numpy(), mo.place(L, st["actions"], world_axis=1))
    assert np.array_equal(buf.action_log_probs.cpu().numpy(), mo.place(L, st["logp"], world_axis=1))
    assert np.array_equal(buf.value_preds[:L].cpu().numpy(), mo.place(L, st["values"], world_axis=1))
    assert np.array_equal(buf.rewards.cpu().numpy(), mo.place(L, st["rewards"], world_axis=1))
    assert np.array_equal(buf.dones.cpu().numpy(), mo.place(L, st["dones"], world_axis=0))
    assert not buf.obs[L].any()
    env.close()


def test_bench_shape_cramped_room():
    """L = 400, 20 replicas (7,980 worlds, 125 tiles), as tools/rollout_bench.py --mode mixed measures it"""
    lp = layouts.load_layout("simple", 100)
    pol, _, _ = make_policies(lp, 2)
    assert_same(run("simple", pol, 400, 20, False, horizon=100), run("simple", pol, 400, 20, True, horizon=100))


def test_graph_replay_equals_direct_launches():
    L, replicas = 7, 20
    N = replicas * (L - 1)
    lp = layouts.load_layout("simple", 400)
    pol, _, _ = make_policies(lp, 2)
    out = []
    for use_graph in (False, True):
        env = B200Overcooked("simple", N, 0, horizon=11, seed=9)
        col = MixedPlayCollector(env, pol, L, 0, 1, seed=3, mix_seed=8, use_graph=use_graph, fused=True)
        assert col._scratch is None
        col.collect()
        b = col.collect()   # the second collection continues from the first one's final state
        torch.cuda.synchronize()
        assert col.fused is True
        out.append([t.clone() for t in (b.obs, b.actions, b.action_log_probs, b.value_preds, b.rewards, b.dones)])
        out[-1].append(torch.from_numpy(env.get_state()))
        out[-1].append(torch.tensor([env.step_count]))
        env.close()
    for a, b in zip(*out):
        assert torch.equal(a.cpu(), b.cpu())


@pytest.mark.parametrize("layout,hidden", [("simple", 512), ("schelling", 64)])
def test_unsupported_handles_fall_back(layout, hidden):
    """hidden 512 and a generic-kernel layout: OCB_ERR_UNSUPPORTED from the C entry point; the collector falls back with
    fused=None (same buffers as fused=False) and raises with fused=True"""
    L, N = 5, 256
    lp = layouts.load_layout(layout, 400)
    pol = FusedPolicy(lp, hidden, 2)
    for i in range(2):
        pol.set_weights(i, PolicyNet("actor", lp.width, lp.height, lp.channels, hidden).init_like_reference(i, gain=2.0),
                        PolicyNet("critic", lp.width, lp.height, lp.channels, hidden).init_like_reference(50 + i))
    lib = _native.lib()
    env = B200Overcooked(layout, N, 0, horizon=400, seed=1)
    buf = MixedPlayBuffer(env, L)
    rc = lib.ocb_rollout_mixed_fused(env._h, pol._h, L, 0, 1, _ptr(buf.obs), _ptr(buf.actions), None, None, None, None,
                                     0, 1, 2, None)
    assert rc == _native.OCB_ERR_UNSUPPORTED and env.step_count == 0
    with pytest.raises(_native.NativeError) as e:
        MixedPlayCollector(env, pol, L, fused=True).collect()
    assert e.value.code == _native.OCB_ERR_UNSUPPORTED
    env.close()
    res = []
    for fused in (None, False):
        env = B200Overcooked(layout, N, 0, horizon=400, seed=1)
        col = MixedPlayCollector(env, pol, L, 0, 1, seed=4, mix_seed=6, fused=fused)
        b = col.collect()
        torch.cuda.synchronize()
        assert col.fused is False
        res.append([t.clone() for t in (b.obs, b.actions, b.action_log_probs, b.value_preds, b.rewards, b.dones)])
        res[-1].append(torch.from_numpy(env.get_state()))
        env.close()
    for a, b in zip(*res):
        assert torch.equal(a.cpu(), b.cpu())


def test_argument_errors_match_the_per_step_entry_point_and_launch_nothing():
    lp = layouts.load_layout("simple", 400)
    pol, _, _ = make_policies(lp, 2)
    lib = _native.lib()
    env = B200Overcooked("simple", 30, 0, horizon=400, seed=1)
    buf = MixedPlayBuffer(env, 7)
    buf.actions.fill_(-7)
    state = env.get_state()
    scratch = torch.empty((int(lib.ocb_rollout_mixed_scratch_bytes(env._h)),), dtype=torch.uint8, device=env.sim_device)
    o, a = _ptr(buf.obs), _ptr(buf.actions)
    cases = [
        ("NULL env", (None, pol._h, 7, 0, 1, o, a)),
        ("NULL policy", (env._h, None, 7, 0, 1, o, a)),
        ("NULL obs_buf", (env._h, pol._h, 7, 0, 1, None, a)),
        ("NULL actions", (env._h, pol._h, 7, 0, 1, o, None)),
        ("L < 2", (env._h, pol._h, 1, 0, 1, o, a)),
        ("N % (L - 1)", (env._h, pol._h, 8, 0, 1, o, a)),
        ("main out of range", (env._h, pol._h, 7, 2, 1, o, a)),
        ("partner out of range", (env._h, pol._h, 7, 0, -1, o, a)),
    ]
    for what, head in cases:
        rest = (None, None, None, None, 0, 0, 0)
        rc = lib.ocb_rollout_mixed_fused(*head, *rest, None)
        msg = lib.ocb_last_error()
        rc_ref = lib.ocb_rollout_mixed(*head, *rest, _ptr(scratch), scratch.numel(), None)
        assert rc == OCB_ERR_INVALID_ARG and rc_ref == OCB_ERR_INVALID_ARG, what
        assert msg == lib.ocb_last_error(), what
    # a misaligned obs_buf is refused before the rollout runs, so no buffer or env state moves
    rc = lib.ocb_rollout_mixed_fused(env._h, pol._h, 7, 0, 1, ctypes.c_void_p(buf.obs.data_ptr() + 1), a,
                                     None, None, None, None, 0, 0, 0, None)
    assert rc == OCB_ERR_INVALID_ARG and b"aligned" in lib.ocb_last_error()
    torch.cuda.synchronize()
    assert bool((buf.actions == -7).all()) and int(buf.obs.abs().sum()) == 0
    assert np.array_equal(env.get_state(), state) and env.step_count == 0
    env.close()
