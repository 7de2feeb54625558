"""GPU tests of the fused tensor-core policy forward (csrc/policy_kernels.cu) through the C ABI.

Numerics: compared with a plain PyTorch fp32 forward of the same network
(diverse_conventions_b200/policy.py: PolicyNet.forward, itself identical to the reference's
R_Actor / R_Critic on the committed golden vectors).  Tolerance of the north star: logits
within 1e-3 relative; the hi/lo bf16 operand split gets ~1e-5, the tests assert 2e-4."""
import os

import numpy as np
import pytest
import torch

from diverse_conventions_b200 import layouts
from diverse_conventions_b200.overcooked_env import B200Overcooked
from diverse_conventions_b200.policy import FusedPolicy, PolicyNet, log_softmax_sample
from oracle.c_oracle import COracle

pytestmark = pytest.mark.gpu

REL_TOL = 2e-4  # max |err| / max |reference| (north star allows 1e-3)


def rel_err(a, b):
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-12))


def golden_nets(golden_dir, layout):
    g = np.load(os.path.join(golden_dir, "policy_%s_h64.npz" % layout))
    lp = layouts.load_layout(layout, 400)
    nets = {}
    for kind in ("actor", "critic"):
        net = PolicyNet(kind, lp.width, lp.height, lp.channels, 64)
        net.load_state_dict({k[len(kind) + 1:]: torch.from_numpy(g[k]) for k in g.files if k.startswith(kind + ".")})
        nets[kind] = net
    return g, lp, nets


@pytest.mark.parametrize("layout", ["simple", "random1"])
def test_matches_reference_networks_on_golden_vectors(golden_dir, layout):
    g, lp, nets = golden_nets(golden_dir, layout)
    pol = FusedPolicy(lp, 64, 1)
    pol.set_weights(0, nets["actor"], nets["critic"])
    obs = torch.from_numpy(g["obs"]).cuda()
    out = pol.act(obs, deterministic=True, want_logits=True)
    val = pol.value(obs)
    torch.cuda.synchronize()
    ref_logits, ref_values = torch.from_numpy(g["logits"]), torch.from_numpy(g["values"])[:, 0]
    assert rel_err(out["logits"].cpu(), ref_logits) < REL_TOL
    assert rel_err(val.cpu(), ref_values) < REL_TOL
    # also element-wise: |err| <= 1e-3 * |ref| + tiny absolute floor
    assert torch.allclose(out["logits"].cpu(), ref_logits, rtol=1e-3, atol=2e-6)
    # arg-max action and its log-prob (FixedCategorical.mode / log_probs)
    lg = out["logits"].cpu()
    assert torch.equal(out["actions"].cpu().long(), lg.argmax(-1))
    assert torch.allclose(out["logp"].cpu(), log_softmax_sample(lg, out["actions"].cpu()), atol=1e-6)


def test_ragged_rows_many_policies_and_tile_selection():
    lp = layouts.load_layout("simple", 400)
    n_pol = 5
    pol = FusedPolicy(lp, 64, n_pol)
    actors = [PolicyNet("actor", 5, 4, 20, 64).init_like_reference(10 + i, gain=1.0) for i in range(n_pol)]
    critics = [PolicyNet("critic", 5, 4, 20, 64).init_like_reference(50 + i) for i in range(n_pol)]
    for i in range(n_pol):
        for net in (actors[i], critics[i]):
            net.conv_b.uniform_(-0.1, 0.1), net.fc1_b.uniform_(-0.1, 0.1), net.fc2_b.uniform_(-0.1, 0.1), net.head_b.uniform_(-0.1, 0.1)
        pol.set_weights(i, actors[i], critics[i])
    # observations from random play (objects, soups, both views)
    N = 700
    orc = COracle(lp, N)
    rng = np.random.default_rng(0)
    for _ in range(150):
        o, _, _ = orc.step(rng.choice(6, size=(2, N), p=[.15, .15, .15, .15, .05, .35]))
    M = 2 * N - 37  # not a multiple of 128
    obs = torch.from_numpy(o.reshape(2 * N, 5, 4, 20)[:M].copy()).cuda()
    tiles = (M + 127) // 128
    tile_policy = torch.tensor([(3 * t + 1) % n_pol for t in range(tiles)], dtype=torch.int32, device="cuda")
    out = pol.act(obs, tile_policy=tile_policy, deterministic=True, want_logits=True)
    val = pol.value(obs, tile_policy=tile_policy)
    torch.cuda.synchronize()
    ref_l = torch.empty((M, 6))
    ref_v = torch.empty((M,))
    for t in range(tiles):
        sl = slice(t * 128, min(M, (t + 1) * 128))
        k = int(tile_policy[t])
        ref_l[sl] = actors[k].forward(obs[sl].cpu())
        ref_v[sl] = critics[k].forward(obs[sl].cpu())[:, 0]
    assert rel_err(out["logits"].cpu(), ref_l) < REL_TOL
    assert rel_err(val.cpu(), ref_v) < REL_TOL


@pytest.mark.parametrize("layout", ["simple", "random1", "unident_s"])
def test_single_network_mode_equals_the_pair_kernel(layout):
    """ocb_policy_act / ocb_policy_value run the pair kernel's one-network mode (both epilogue groups on one stream): every
    output element sums the same products in the same order as the two-network forward, so logits and values are
    BIT-identical to ocb_policy_forward.  Several weight sets per launch (tile_policy), ragged row count."""
    lp = layouts.load_layout(layout, 400)
    n_pol, N = 3, 900
    nets = [(PolicyNet("actor", lp.width, lp.height, lp.channels, 64).init_like_reference(3 + i, gain=1.0),
             PolicyNet("critic", lp.width, lp.height, lp.channels, 64).init_like_reference(40 + i)) for i in range(n_pol)]
    orc, rng = COracle(lp, N), np.random.default_rng(5)
    for _ in range(60):
        o, _, _ = orc.step(rng.choice(6, size=(2, N), p=[.15, .15, .15, .15, .05, .35]))
    M = 2 * N - 61
    obs = torch.from_numpy(o.reshape(2 * N, lp.width, lp.height, lp.channels)[:M].copy()).cuda()
    tiles = (M + 127) // 128
    tile_policy = torch.tensor([(2 * t + 1) % n_pol for t in range(tiles)], dtype=torch.int32, device="cuda")

    pol = FusedPolicy(lp, 64, n_pol)
    for i, (a, c) in enumerate(nets):
        pol.set_weights(i, a, c)
    act = pol.act(obs, tile_policy=tile_policy, seed=9, offset=4, want_logits=True)
    val = pol.value(obs, tile_policy=tile_policy)
    both = pol.forward(obs, tile_policy=tile_policy, seed=9, offset=4, want_logits=True)
    torch.cuda.synchronize()
    assert torch.equal(act["logits"], both["logits"]) and torch.equal(val, both["values"])
    assert torch.equal(act["actions"], both["actions"]) and torch.equal(act["logp"], both["logp"])
    pol.close()


def test_sampling_follows_the_softmax_and_is_reproducible():
    lp = layouts.load_layout("simple", 400)
    pol = FusedPolicy(lp, 64, 1)
    actor = PolicyNet("actor", 5, 4, 20, 64).init_like_reference(4, gain=3.0)  # peaked enough to test
    pol.set_weights(0, actor, PolicyNet("critic", 5, 4, 20, 64).init_like_reference(5))
    one = torch.from_numpy(COracle(lp, 1).observe()[0]).cuda()  # reset observation of player 0
    M = 1 << 16
    obs = one.expand(M, 5, 4, 20).contiguous()
    a = pol.act(obs, seed=7, offset=3, want_logits=True)
    b = pol.act(obs, seed=7, offset=3)
    c = pol.act(obs, seed=7, offset=4)
    assert torch.equal(a["actions"], b["actions"]) and not torch.equal(a["actions"], c["actions"])
    probs = torch.softmax(a["logits"][0].cpu().double(), -1)
    freq = torch.bincount(a["actions"].cpu().long(), minlength=6).double() / M
    assert float((freq - probs).abs().max()) < 4.5 * float(torch.sqrt(probs * (1 - probs) / M).max())
    assert torch.allclose(a["logp"].cpu(), log_softmax_sample(a["logits"].cpu(), a["actions"].cpu()), atol=1e-6)


def test_unsupported_shapes_fail_loudly():
    from diverse_conventions_b200 import _native
    with pytest.raises(_native.NativeError):
        FusedPolicy(layouts.load_layout("simple", 400), hidden=128)


@pytest.mark.parametrize("hidden", [64, 512])
@pytest.mark.parametrize("layout,N", [("schelling", 75), ("multiplayer_schelling", 41), ("corridor", 30), ("simple_single", 130)])
def test_shapes_outside_the_tensor_core_range_run_the_generic_kernel(layout, N, hidden):
    """7- and 9-row grids, 4 players (30 channels, rows of 1,470 bytes) and 1 player: the reference's CNNBase takes any
    shape (train/MAPPO/utils/cnn.py:22-42); here they run policy_generic_kernel behind the same entry points"""
    lp = layouts.load_layout(layout, 400)
    actor = PolicyNet("actor", lp.width, lp.height, lp.channels, hidden).init_like_reference(3, gain=1.5)
    critic = PolicyNet("critic", lp.width, lp.height, lp.channels, hidden).init_like_reference(4)
    for net in (actor, critic):
        for b in (net.conv_b, net.fc1_b, net.fc2_b, net.head_b):
            b.uniform_(-0.1, 0.1)
    pol = FusedPolicy(lp, hidden, 2)
    pol.set_weights(1, actor, critic)
    from oracle.c_oracle import COracle
    orc = COracle(lp, N)
    rng = np.random.default_rng(1)
    for _ in range(40):
        o, _, _ = orc.step(rng.integers(0, 6, size=(lp.num_players, N)))
    obs = torch.from_numpy(o.reshape(-1, lp.width, lp.height, lp.channels).copy()).cuda()
    M = obs.shape[0]
    tiles = torch.ones(((M + 127) // 128,), dtype=torch.int32, device="cuda")
    out = pol.forward(obs, tile_policy=tiles, deterministic=True, want_logits=True)
    torch.cuda.synchronize()
    ref_l, ref_v = actor.forward(obs.cpu()), critic.forward(obs.cpu())[:, 0]
    assert torch.allclose(out["logits"].cpu(), ref_l, rtol=1e-4, atol=1e-5)
    assert torch.allclose(out["values"].cpu(), ref_v, rtol=1e-4, atol=1e-5)
    assert torch.equal(out["actions"].cpu().long(), out["logits"].cpu().argmax(-1))
    a = pol.act(obs, tile_policy=tiles, seed=3, offset=9, want_logits=True)
    assert torch.allclose(a["logp"].cpu(), log_softmax_sample(a["logits"].cpu(), a["actions"].cpu()), atol=1e-6)
    assert torch.equal(pol.value(obs, tile_policy=tiles), out["values"])


def test_generic_kernel_agrees_with_the_tensor_core_kernels(monkeypatch):
    """the same handle shape through both paths (OCB_POLICY_GENERIC=1 forces the generic kernel): same sampled actions,
    logits within the tensor-core path's tolerance"""
    lp = layouts.load_layout("random1", 400)
    actor = PolicyNet("actor", lp.width, lp.height, lp.channels, 64).init_like_reference(8, gain=2.0)
    critic = PolicyNet("critic", lp.width, lp.height, lp.channels, 64).init_like_reference(9)
    env = B200Overcooked("random1", 300, 0, horizon=400, seed=2)
    obs = env.rollout_random(25)["obs"][-1].contiguous()
    tc = FusedPolicy(lp, 64, 1)
    tc.set_weights(0, actor, critic)
    monkeypatch.setenv("OCB_POLICY_GENERIC", "1")
    gen = FusedPolicy(lp, 64, 1)
    gen.set_weights(0, actor, critic)
    a = tc.forward(obs, seed=5, offset=2, want_logits=True)
    b = gen.forward(obs, seed=5, offset=2, want_logits=True)
    assert torch.allclose(a["logits"], b["logits"], rtol=2e-4, atol=2e-5) and torch.allclose(a["values"], b["values"], rtol=2e-4, atol=2e-5)
    assert float((a["actions"] == b["actions"]).float().mean()) > 0.999  # same counters; ties in the inverse CDF aside


@pytest.mark.parametrize("layout", ["simple", "random0", "random3", "unident_s", "scenario3"])
def test_fused_forward_all_layout_sizes(layout):
    """both networks in one launch, weights resident (small grids) or streamed (large grids);
    enough rows that every CTA runs several tiles back to back"""
    lp = layouts.load_layout(layout, 400)
    n_pol = 3
    pol = FusedPolicy(lp, 64, n_pol)
    actors = [PolicyNet("actor", lp.width, lp.height, 20, 64).init_like_reference(20 + i, gain=1.0) for i in range(n_pol)]
    critics = [PolicyNet("critic", lp.width, lp.height, 20, 64).init_like_reference(70 + i) for i in range(n_pol)]
    for i in range(n_pol):
        for net in (actors[i], critics[i]):
            for b in (net.conv_b, net.fc1_b, net.fc2_b, net.head_b):
                b.uniform_(-0.1, 0.1)
        pol.set_weights(i, actors[i], critics[i])
    N = 148 * 64 * 2 + 77
    orc = COracle(lp, N)
    rng = np.random.default_rng(1)
    for _ in range(60):
        o, _, _ = orc.step(rng.choice(6, size=(2, N), p=[.15, .15, .15, .15, .05, .35]))
    M = 2 * N
    obs = torch.from_numpy(o.reshape(M, lp.width, lp.height, 20).copy()).cuda()
    tiles = (M + 127) // 128
    for tp in (None, torch.tensor([(t // 5) % n_pol for t in range(tiles)], dtype=torch.int32, device="cuda")):
        out = pol.forward(obs, tile_policy=tp, deterministic=True, want_logits=True)
        torch.cuda.synchronize()
        pick = torch.arange(0, tiles, 7)
        for t in pick.tolist() + [tiles - 1]:
            sl = slice(t * 128, min(M, (t + 1) * 128))
            k = 0 if tp is None else int(tp[t])
            assert rel_err(out["logits"][sl].cpu(), actors[k].forward(obs[sl].cpu())) < REL_TOL, (layout, t)
            assert rel_err(out["values"][sl].cpu(), critics[k].forward(obs[sl].cpu())[:, 0]) < REL_TOL, (layout, t)
        # the single-network entry points run the pair kernel's single mode: same products in the same order
        a = pol.act(obs, tile_policy=tp, deterministic=True, want_logits=True)
        v = pol.value(obs, tile_policy=tp)
        assert torch.equal(a["logits"], out["logits"])
        assert torch.equal(a["actions"], out["actions"])
        assert torch.equal(v, out["values"])
    info = pol.info()
    assert info["ring_slots"] >= 4 and info["smem_bytes"] <= 227 * 1024
