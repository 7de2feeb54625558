"""Device-side weight refresh (ocb_policy_set_weights_device / FusedPolicy.set_weights_device).

The device path must leave the handle exactly as the host path (ocb_policy_set_weights) leaves it: the packed blobs byte
for byte in all three formats (hidden-64 tensor-core, hidden-512, generic fp32 kernel), the forward outputs bit for bit,
and the critic's zero-observation value that mixed play writes to slot L.  The refresh is stream-ordered and, given to a
collector as ``weights=``, part of its CUDA graph: a replay after an in-place parameter update (as an optimizer step makes)
collects with the new parameters.  The last tests cover the argument errors, after which the blobs are untouched.
"""
import ctypes

import pytest
import torch

from diverse_conventions_b200 import _native, layouts
from diverse_conventions_b200.mixed import MixedPlayCollector
from diverse_conventions_b200.overcooked_env import B200Overcooked
from diverse_conventions_b200.policy import FusedPolicy, PolicyNet
from diverse_conventions_b200.rollout import PolicyRollout, crossplay_training_tables, pair_tile_policy

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda", 0)


def special_values(t, g):
    """overwrite ~3 % of t with values the bf16 hi/lo split must round alike on both paths: exact bf16 rounding ties (and
    their neighbours), subnormals, +-0 and large magnitudes"""
    n = t.numel()
    k = min(n, max(8, n // 32))
    idx = torch.randperm(n, generator=g)[:k]
    hi = torch.randint(0, 1 << 16, (k,), generator=g, dtype=torch.int64) & 0x7F7F  # finite exponents only
    sign = torch.randint(0, 2, (k,), generator=g, dtype=torch.int64) << 31
    low = torch.tensor([0x8000, 0x7FFF, 0x8001, 0x8000], dtype=torch.int64)[torch.randint(0, 4, (k,), generator=g)]
    bits = sign | (hi << 16) | low
    kind = torch.randint(0, 5, (k,), generator=g)
    bits = torch.where(kind == 1, sign | torch.randint(1, 1 << 23, (k,), generator=g, dtype=torch.int64), bits)  # subnormal
    bits = torch.where(kind == 2, sign, bits)  # +-0
    big = torch.tensor(3.0e4).view(torch.int32).item()
    bits = torch.where(kind == 3, sign | (big + torch.randint(0, 1 << 20, (k,), generator=g, dtype=torch.int64)), bits)
    vals = bits.to(torch.int32).view(torch.float32)
    flat = t.view(-1)
    flat[idx] = vals
    return t


def random_net(kind, lp, hidden, seed, device="cpu"):
    g = torch.Generator().manual_seed(seed)
    net = PolicyNet(kind, lp.width, lp.height, lp.channels, hidden)
    for name in ("conv_w", "conv_b", "fc1_w", "fc1_b", "fc2_w", "fc2_b", "head_w", "head_b"):
        t = getattr(net, name)
        t.copy_(torch.randn(t.shape, generator=g) * (0.5 / max(1, t.shape[-1]) ** 0.5 if t.dim() > 1 else 0.1))
        special_values(t, g)
    if device != "cpu":
        net = on_device(net, device)
    return net


def on_device(net, device=DEV):
    """a copy of `net` whose tensors live on the device, made the way a trainer's module would be aliased"""
    d = PolicyNet(net.kind, net.W, net.H, net.C, net.hidden, device=device)
    return d.alias_state_dict({k: v.to(device).contiguous() for k, v in net.state_dict().items()})


def on_host(net):
    h = PolicyNet(net.kind, net.W, net.H, net.C, net.hidden)
    return h.load_state_dict({k: v.cpu() for k, v in net.state_dict().items()})


def make_handle(lp, hidden, n):
    try:
        return FusedPolicy(lp, hidden, n)
    except _native.NativeError as e:
        if e.code == _native.OCB_ERR_UNSUPPORTED:
            pytest.skip("the handle does not take %s at hidden %d" % (lp.name if hasattr(lp, "name") else lp, hidden))
        raise


def blobs(pol):
    torch.cuda.synchronize()
    return [pol.read_blob(i, net).clone() for i in range(pol.n_policies) for net in (0, 1)]


def bits_equal(a, b):
    if a is None or b is None:
        return a is None and b is None
    if a.dtype == torch.float32:
        return torch.equal(a.view(torch.int32), b.view(torch.int32))
    return torch.equal(a, b)


def real_observations(layout, rows):
    """`rows` observation rows of random play on `layout` (int8 [rows, W, H, C])"""
    env = B200Overcooked(layout, 4096, 0, horizon=50, seed=3)
    per = env.num_players * env.num_envs
    out = env.rollout_random((rows + per - 1) // per)
    obs = out["obs"].reshape(-1, env.width, env.height, env.channels)[:rows].contiguous()
    torch.cuda.synchronize()
    env.close()
    return obs


# ---------------------------------------------------------------------------- byte identity
@pytest.mark.parametrize("hidden", [64, 512])
@pytest.mark.parametrize("layout", ["cramped_room", "coordination_ring", "counter_circuit", "asymmetric_advantages",
                                    "schelling", "simple_single"])
def test_device_refresh_writes_the_host_paths_bytes_and_forward(layout, hidden):
    lp = layouts.load_layout(layout, 400)
    host, dev = make_handle(lp, hidden, 2), make_handle(lp, hidden, 2)
    nets = [(random_net("actor", lp, hidden, 10 + i), random_net("critic", lp, hidden, 20 + i)) for i in range(2)]
    other = [(random_net("actor", lp, hidden, 30 + i), random_net("critic", lp, hidden, 40 + i)) for i in range(2)]
    for i, (a, c) in enumerate(nets):
        host.set_weights(i, a, c)
    for i, (a, c) in enumerate(other):  # whatever the device path overwrites must not show through
        dev.set_weights(i, a, c)
    dev.set_weights_device([(i, on_device(a), on_device(c)) for i, (a, c) in enumerate(nets)])
    for k, (x, y) in enumerate(zip(blobs(host), blobs(dev))):
        assert torch.equal(x, y), "blob %d differs at %s" % (k, torch.nonzero(x != y)[:8].flatten().tolist())

    obs = real_observations(layout, 32768)
    M = obs.shape[0]
    tiles = (M + 127) // 128
    table = (torch.arange(tiles, dtype=torch.int32, device=DEV) % 2).contiguous()
    acts = torch.randint(0, 6, (M,), dtype=torch.int32, device=DEV)
    outs = []
    for pol in (host, dev):
        o = {"forward": pol.forward(obs, table, seed=5, offset=3, want_logits=True),
             "act": pol.act(obs, table, seed=6, offset=1, want_logits=True),
             "value": {"values": pol.value(obs, table)},
             "evaluate": pol.evaluate(obs, acts, tile_policy=table, want_logits=True)}
        torch.cuda.synchronize()
        outs.append(o)
    for name in outs[0]:
        for key, x in outs[0][name].items():
            assert bits_equal(x, outs[1][name][key]), (name, key)


# ---------------------------------------------------------------------------- many sets, partial refreshes
def test_sixteen_sets_in_one_call_and_partial_refreshes():
    lp = layouts.load_layout("cramped_room", 400)
    host, dev = make_handle(lp, 64, 16), make_handle(lp, 64, 16)
    nets = [(random_net("actor", lp, 64, 100 + i), random_net("critic", lp, 64, 200 + i)) for i in range(16)]
    for i, (a, c) in enumerate(nets):
        host.set_weights(i, a)
        host.set_weights(i, critic=c)
    dev.set_weights_device([(i, on_device(a), on_device(c)) for i, (a, c) in enumerate(nets)])
    before = blobs(dev)
    assert all(torch.equal(x, y) for x, y in zip(blobs(host), before))

    # only the actor of some sets, only the critic of others: every other blob keeps its bytes
    new_a = {3: random_net("actor", lp, 64, 300), 9: random_net("actor", lp, 64, 301)}
    new_c = {7: random_net("critic", lp, 64, 302), 9: random_net("critic", lp, 64, 303)}
    sets = [(3, on_device(new_a[3]), None), (7, None, on_device(new_c[7])), (9, on_device(new_a[9]), on_device(new_c[9]))]
    dev.set_weights_device(sets)
    for i, net in new_a.items():
        host.set_weights(i, actor=net)
    for i, net in new_c.items():
        host.set_weights(i, critic=net)
    after, want = blobs(dev), blobs(host)
    changed = {(3, 0), (7, 1), (9, 0), (9, 1)}
    for k, (x, y, b) in enumerate(zip(after, want, before)):
        assert torch.equal(x, y), k
        if (k // 2, k % 2) not in changed:
            assert torch.equal(x, b), k


# ---------------------------------------------------------------------------- stream order
def snapshot(buf):
    return [None if t is None else t.clone() for t in (buf.obs, buf.actions, buf.action_log_probs, buf.value_preds,
                                                       buf.rewards, buf.dones)]


def assert_buffers_equal(a, b):
    for name, x, y in zip(("obs", "actions", "logp", "values", "rewards", "dones"), a, b):
        assert bits_equal(x, y), name


def test_refresh_is_ordered_between_two_collections():
    lp = layouts.load_layout("coordination_ring", 400)
    A = [random_net("actor", lp, 64, 1), random_net("critic", lp, 64, 2)]
    B = [random_net("actor", lp, 64, 3), random_net("critic", lp, 64, 4)]
    Bd = [on_device(n) for n in B]
    T, N = 40, 2048

    env = B200Overcooked("coordination_ring", N, 0, horizon=30, seed=8)
    pol = make_handle(lp, 64, 1)
    pol.set_weights(0, *A)
    ro = PolicyRollout(env, pol, T, seed=5)
    torch.cuda.synchronize()
    first = snapshot(ro.collect())  # clones are stream-ordered: nothing synchronises until the end
    pol.set_weights_device([(0, Bd[0], Bd[1])])
    second = snapshot(ro.collect())
    torch.cuda.synchronize()

    env2 = B200Overcooked("coordination_ring", N, 0, horizon=30, seed=8)
    pol2 = make_handle(lp, 64, 1)
    pol2.set_weights(0, *A)
    ro2 = PolicyRollout(env2, pol2, T, seed=5)
    want1 = snapshot(ro2.collect())
    torch.cuda.synchronize()
    pol2.set_weights(0, *B)
    want2 = snapshot(ro2.collect())
    torch.cuda.synchronize()
    assert_buffers_equal(first, want1)
    assert_buffers_equal(second, want2)
    assert not torch.equal(want1[3], want2[3])


# ---------------------------------------------------------------------------- graph replay with weights=
def trainer_nets(lp, hidden, n, seed):
    """per weight set an (actor, critic) pair of device nets aliasing 'trainer' parameters (the dicts returned too)"""
    out = []
    for i in range(n):
        pair = []
        for kind, s in (("actor", seed + i), ("critic", seed + 100 + i)):
            src = PolicyNet(kind, lp.width, lp.height, lp.channels, hidden).init_like_reference(s, gain=2.0 if kind == "actor" else 1.0)
            for b in (src.conv_b, src.fc1_b, src.fc2_b, src.head_b):
                b.uniform_(-0.1, 0.1, generator=torch.Generator().manual_seed(s))
            params = {k: v.to(DEV).clone() for k, v in src.state_dict().items()}
            pair.append(PolicyNet(kind, lp.width, lp.height, lp.channels, hidden, device=DEV).alias_state_dict(params))
        out.append(tuple(pair))
    return out


def optimizer_step(nets, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    for pair in nets:
        for net in pair:
            for t in net.state_dict().values():
                t.add_(torch.randn(t.shape, generator=g, device=DEV) * 0.05)


def collector(mode, env, pol, weights=None, use_graph=False, hidden=64):
    if mode == "mixed":
        return MixedPlayCollector(env, pol, 9, seed=3, mix_seed=11, use_graph=use_graph, weights=weights)
    kw = {}
    if mode == "crossplay_train":
        slices = [((0, 0), (0, 0)), ((0, 1), (1, None)), ((1, None), (0, 2)), ((2, None), (2, None))]
        tp, cp = crossplay_training_tables(slices, 256, DEV)
        kw = dict(tile_policy=tp, critic_policy=cp)
    elif mode == "population":
        kw = dict(tile_policy=pair_tile_policy([(0, 0), (1, 1), (2, 2), (1, 1)], 256, DEV))
    return PolicyRollout(env, pol, 24, seed=3, use_graph=use_graph, weights=weights, **kw)


@pytest.mark.parametrize("mode,hidden", [("selfplay", 64), ("selfplay", 512), ("crossplay_train", 64), ("population", 64),
                                         ("mixed", 64), ("mixed", 512)])
def test_graph_replay_collects_with_the_parameters_of_the_moment(mode, hidden):
    lp = layouts.load_layout("cramped_room", 400)
    n = 1 if mode == "selfplay" else 3
    N = 8 * 128 if mode != "mixed" else 8 * 120
    nets = trainer_nets(lp, hidden, n, 60)
    sets = [(i, a, c) for i, (a, c) in enumerate(nets)]

    env_g = B200Overcooked("cramped_room", N, 0, horizon=20, seed=4)
    env_d = B200Overcooked("cramped_room", N, 0, horizon=20, seed=4)
    pol_g, pol_d = make_handle(lp, hidden, n), make_handle(lp, hidden, n)
    col_g = collector(mode, env_g, pol_g, weights=sets, use_graph=True)
    col_d = collector(mode, env_d, pol_d)
    for step in range(3):
        got = snapshot(col_g.collect())
        for i, (a, c) in enumerate(nets):
            pol_d.set_weights(i, on_host(a), on_host(c))
        want = snapshot(col_d.collect())
        torch.cuda.synchronize()
        assert_buffers_equal(got, want)
        optimizer_step(nets, 1000 + step)


# ---------------------------------------------------------------------------- slot L of mixed play under graph replay
@pytest.mark.parametrize("hidden", [64, 512])
def test_mixed_graph_replay_bootstraps_from_the_current_critic(hidden):
    """values[L] is the zero-observation value of main's critic as loaded at replay time, not at capture time (a graph
    used to capture the value as a launch argument, so host set_weights between replays left it stale)"""
    lp = layouts.load_layout("cramped_room", 400)
    L, N = 9, 8 * 120
    a0, a1 = [PolicyNet("actor", lp.width, lp.height, lp.channels, hidden).init_like_reference(s, gain=2.0) for s in (1, 2)]
    c_old, c_new = [PolicyNet("critic", lp.width, lp.height, lp.channels, hidden).init_like_reference(s) for s in (3, 4)]
    for c in (c_old, c_new):  # a clearly non-zero value of the zero observation
        c.conv_b.uniform_(0.0, 0.2, generator=torch.Generator().manual_seed(7))
        c.fc1_b.uniform_(-0.1, 0.1, generator=torch.Generator().manual_seed(8))
        c.head_b.fill_(0.25)
    pol = make_handle(lp, hidden, 2)
    pol.set_weights(0, a0, c_old)
    pol.set_weights(1, a1)
    col = MixedPlayCollector(B200Overcooked("cramped_room", N, 0, horizon=20, seed=4), pol, L, use_graph=True)
    old = col.collect().value_preds[L].clone()
    pol.set_weights(0, critic=c_new)
    new = col.collect().value_preds[L].clone()

    ref = make_handle(lp, hidden, 2)  # the host path's value of c_new, through a direct collection
    ref.set_weights(0, a0, c_new)
    ref.set_weights(1, a1)
    want = MixedPlayCollector(B200Overcooked("cramped_room", N, 0, horizon=20, seed=4), ref, L).collect().value_preds[L]
    torch.cuda.synchronize()
    zero = torch.zeros((1, lp.width, lp.height, lp.channels))
    assert torch.allclose(want[0, 0].cpu(), c_new.forward(zero)[0, 0], rtol=1e-4, atol=1e-5)
    assert not torch.equal(old, want)
    assert bits_equal(new, want)


# ---------------------------------------------------------------------------- errors
def srcs(pol, sets):
    return pol._weight_srcs(sets)


def call(pol_h, n, arr):
    return _native.lib().ocb_policy_set_weights_device(pol_h, n, arr, None)


def test_rejected_calls_launch_nothing():
    lib = _native.lib()
    lp = layouts.load_layout("cramped_room", 400)
    pol = make_handle(lp, 64, 2)
    nets = [(random_net("actor", lp, 64, 1 + i), random_net("critic", lp, 64, 5 + i)) for i in range(2)]
    for i, (a, c) in enumerate(nets):
        pol.set_weights(i, a, c)
    before = blobs(pol)
    fresh = [(on_device(random_net("actor", lp, 64, 50)), on_device(random_net("critic", lp, 64, 51)))]

    def rejected(n, arr, words):
        rc = call(pol._h, n, arr)
        assert rc == -1, rc
        msg = lib.ocb_last_error().decode()
        assert all(w in msg for w in words), msg

    good = srcs(pol, [(0, fresh[0][0], fresh[0][1])])
    assert call(None, 2, good) == -1
    rejected(2, None, ["NULL"])
    rejected(0, good, ["n must be"])
    rejected(-3, good, ["n must be"])
    for field, value, words in (("policy", 2, ["policy 2"]), ("policy", -1, ["policy -1"]), ("net", 2, ["net 2"]),
                                ("net", -1, ["net -1"])):
        arr = srcs(pol, [(0, fresh[0][0], fresh[0][1])])
        setattr(arr[1], field, value)  # the second descriptor is bad: the first must not be packed either
        rejected(2, arr, words)
    arr = srcs(pol, [(0, fresh[0][0], fresh[0][1])])
    arr[1].net = 0
    rejected(2, arr, ["twice"])
    host_t = torch.zeros(64 * 64)
    pinned = torch.zeros(64 * 64).pin_memory()
    for name in ("conv_w", "fc1_b", "head_b"):
        for value, words in ((None, ["NULL", name]), (getattr(arr[1], name) + 2, ["aligned", name]),
                             (host_t.data_ptr(), ["device memory", name]), (pinned.data_ptr(), ["device memory", name])):
            arr = srcs(pol, [(0, fresh[0][0], fresh[0][1])])
            setattr(arr[1], name, value)
            rejected(2, arr, words)
    torch.cuda.synchronize()
    for x, y in zip(before, blobs(pol)):
        assert torch.equal(x, y)


def test_python_side_checks():
    lp = layouts.load_layout("cramped_room", 400)
    pol = make_handle(lp, 64, 2)
    net = PolicyNet("actor", lp.width, lp.height, lp.channels, 64, device=DEV)
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    bad_shape = dict(sd, **{"base.cnn.cnn.3.weight": torch.zeros((64, 10), device=DEV)})
    bad_dtype = dict(sd, **{"base.cnn.cnn.5.weight": sd["base.cnn.cnn.5.weight"].double()})
    bad_contig = dict(sd, **{"base.cnn.cnn.5.weight": sd["base.cnn.cnn.5.weight"].t()})
    bad_device = dict(sd, **{"base.cnn.cnn.0.bias": sd["base.cnn.cnn.0.bias"].cpu()})
    for bad in (bad_shape, bad_dtype, bad_contig, bad_device):
        with pytest.raises(ValueError):
            PolicyNet("actor", lp.width, lp.height, lp.channels, 64, device=DEV).alias_state_dict(bad)
    aliased = PolicyNet("actor", lp.width, lp.height, lp.channels, 64, device=DEV).alias_state_dict(sd)
    sd["base.cnn.cnn.0.weight"].add_(1.0)  # an aliased net sees in-place updates
    assert torch.equal(aliased.conv_w, sd["base.cnn.cnn.0.weight"])

    before = blobs(pol)
    other = layouts.load_layout("coordination_ring", 400)
    wrong_layout = PolicyNet("actor", other.width, other.height, other.channels, 64, device=DEV)
    host_net = PolicyNet("actor", lp.width, lp.height, lp.channels, 64)
    ok = PolicyNet("actor", lp.width, lp.height, lp.channels, 64, device=DEV)
    bent = PolicyNet("actor", lp.width, lp.height, lp.channels, 64, device=DEV)
    bent.fc2_w = bent.fc2_w.t()
    half = PolicyNet("actor", lp.width, lp.height, lp.channels, 64, device=DEV)
    half.head_b = half.head_b.half()
    for sets in ([(0, wrong_layout, None)], [(0, host_net, None)], [(0, bent, None)], [(0, half, None)], [(2, ok, None)],
                 [(0, None, None)], [(1, ok, None), (0, None, ok)]):
        with pytest.raises(ValueError):
            pol.set_weights_device(sets)
    with pytest.raises(ValueError):
        PolicyRollout(B200Overcooked("cramped_room", 256, 0), pol, 4, weights=[(0, wrong_layout, None)])
    for x, y in zip(before, blobs(pol)):
        assert torch.equal(x, y)
