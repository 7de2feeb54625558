"""Device-resident self-play / cross-play rollouts (``ocb_rollout_policy``).

Replaces the host-driven rollout half of the reference trainers:

* ``MainPlayer.collect_episode`` / ``next_step`` (train/MAPPO/main_player.py:91-112, 211-261)
  with the partner seat of ``CentralizedAgent.get_action`` (train/partner_agents.py:28-63):
  per env step 2 actor + 2 critic forwards, ~40 torch launches and a D2H sync on dones.  Here a
  T-step rollout is 2T+1 launches issued from C (or ONE CUDA-graph launch) and nothing
  synchronises; per-world episode returns are accumulated on the device.
* the slice-wise policy multiplexing of ``XDPlayer.next_step`` (train/XD/xd_player.py:177-230) /
  ``CentralizedMultiAgent`` (train/partner_agents.py:87-137): contiguous world slices are driven
  by different (seat-0 policy, seat-1 policy) pairs through a per-128-row ``tile_policy`` table.

The kernels write straight into the PPO rollout buffer.  The buffer is kept SEAT-MAJOR
(``[T(+1), P, N, ...]``, the env's native layout, so every store is contiguous);
``RolloutBuffer.shared_buffer_views()`` exposes it with the axis order of the reference's
``SharedReplayBuffer`` (train/MAPPO/utils/shared_buffer.py:45-76: ``[T(+1), N, P, ...]``) as
zero-copy permuted views, observations stay int8 (the reference stores two fp32 copies).
"""
from __future__ import annotations

import ctypes
from typing import Dict, Optional, Sequence

import torch

from . import _native
from .overcooked_env import B200Overcooked, _ptr
from .policy import FusedPolicy

TILE = FusedPolicy.TILE


class RolloutBuffer:
    """Seat-major PPO rollout storage on the device (one allocation per field)."""

    def __init__(self, env: B200Overcooked, T: int, with_critic: bool = True, with_logp: bool = True):
        P, N, dev = env.num_players, env.num_envs, env.sim_device
        self.T, self.P, self.N = T, P, N
        self.obs = torch.empty((T + 1, P, N, env.width, env.height, env.channels), dtype=torch.int8, device=dev)
        self.actions = torch.empty((T, P, N), dtype=torch.int32, device=dev)
        self.action_log_probs = torch.empty((T, P, N), dtype=torch.float32, device=dev) if with_logp else None
        self.value_preds = torch.empty((T + 1, P, N), dtype=torch.float32, device=dev) if with_critic else None
        self.rewards = torch.empty((T, P, N), dtype=torch.int32, device=dev)
        self.dones = torch.empty((T, N), dtype=torch.int32, device=dev)

    def nbytes(self) -> int:
        return sum(t.numel() * t.element_size() for t in
                   (self.obs, self.actions, self.action_log_probs, self.value_preds, self.rewards, self.dones)
                   if t is not None)

    def compute_returns(self, gamma: float = 0.99, gae_lambda: float = 0.95, use_gae: bool = True, value_normalizer=None,
                        normalize: bool = True, group=None):
        """returns [T+1,P,N] and (normalised) advantages [T,P,N] of this rollout, on the device
        (SharedReplayBuffer.compute_returns + the advantage normalisation of R_MAPPO.train; see returns.py)"""
        from .returns import compute_returns
        if self.value_preds is None:
            raise ValueError("this buffer was collected without the critic")
        self.returns, self.advantages = compute_returns(
            self.value_preds, self.rewards, self.dones, gamma, gae_lambda, use_gae, value_normalizer, normalize,
            getattr(self, "returns", None), getattr(self, "advantages", None), group)
        return self.returns, self.advantages

    def shared_buffer_views(self, hidden_size: int = 64, recurrent_N: int = 1) -> Dict[str, torch.Tensor]:
        """All 13 tensors of the reference's ``SharedReplayBuffer`` (train/MAPPO/utils/shared_buffer.py:45-76), with its
        names, shapes and axis order ``[T(+1), N, P, ...]``, as views of this buffer — nothing is copied except the
        [T+1, N] mask plane.  Field by field, as ``MainPlayer.collect_episode`` + ``chooseinsert`` leave them
        (main_player.py:91-112,211-261, shared_buffer.py:115-148):

        * ``obs`` / ``share_obs``  [T+1,N,P,W,H,C]  the int8 planes (the reference stores two fp32 copies; state == obs,
          envs/overcooked2_env.py:110).  Slot T is the observation after the last step, which the reference only reads
          for the bootstrap value (main_player.py:289-293).
        * ``actions`` / ``action_log_probs`` / ``rewards``  [T,N,P,1]; ``value_preds`` [T+1,N,P,1] (slot T = bootstrap
          value; the reference computes it in ``compute`` instead of storing it).
        * ``masks`` [T+1,N,P,1]: ``masks[t+1] = 1 - done[t]``; ``masks[0] = 1`` as ``reset_after_update`` leaves it
          (shared_buffer.py:240-245; MainPlayer.train calls it after every update).
        * ``bad_masks`` / ``active_masks`` all ones (no time-limit bookkeeping; both seats act every step),
          ``available_actions`` all ones [T+1,N,P,6] (overcooked2_env.py:64), ``rnn_states`` / ``rnn_states_critic``
          zeros [T+1,N,P,recurrent_N,hidden] (feed-forward policies) — broadcast views of one scalar.
        * ``returns`` [T+1,N,P,1]: filled by ``compute_returns`` (zeros before).
        ``masks_next`` (= ``masks[1:]``) is kept for callers of the first version of this method."""
        T, N, P, dev = self.T, self.N, self.P, self.obs.device
        sw = lambda t: None if t is None else t.transpose(1, 2)  # [*, P, N, ...] -> [*, N, P, ...]
        col = lambda t: None if t is None else sw(t).unsqueeze(-1)
        obs = sw(self.obs)
        masks = torch.ones((T + 1, N), dtype=torch.float32, device=dev)
        torch.sub(1.0, self.dones, out=masks[1:])
        masks = masks[:, :, None, None].expand(T + 1, N, P, 1)
        one = torch.ones((), dtype=torch.float32, device=dev)
        zero = torch.zeros((), dtype=torch.float32, device=dev)
        returns = getattr(self, "returns", None)
        return {
            "obs": obs, "share_obs": obs,
            "rnn_states": zero.expand(T + 1, N, P, recurrent_N, hidden_size),
            "rnn_states_critic": zero.expand(T + 1, N, P, recurrent_N, hidden_size),
            "value_preds": col(self.value_preds),
            "returns": col(returns) if returns is not None else zero.expand(T + 1, N, P, 1),
            "available_actions": one.expand(T + 1, N, P, 6),
            "actions": col(self.actions),
            "action_log_probs": col(self.action_log_probs),
            "rewards": col(self.rewards),
            "masks": masks, "bad_masks": one.expand(T + 1, N, P, 1), "active_masks": one.expand(T + 1, N, P, 1),
            "masks_next": masks[1:],
        }

    def fill_shared_replay_buffer(self, shared_buffer):
        """Copy this rollout into an instance of the reference's ``SharedReplayBuffer`` (or anything with its 13 tensor
        attributes), casting to its fp32 storage, so that the reference's ``compute_returns`` /
        ``feed_forward_generator`` / ``R_MAPPO.train`` (shared_buffer.py:248-366, r_mappo.py:166-224) consume a
        device-collected rollout unchanged.  One ``copy_`` per field; the buffer must be ``[T(+1), N, P, ...]``."""
        views = self.shared_buffer_views(int(shared_buffer.rnn_states.shape[-1]), int(shared_buffer.rnn_states.shape[-2]))
        for name in ("share_obs", "obs", "rnn_states", "rnn_states_critic", "value_preds", "returns", "available_actions",
                     "actions", "action_log_probs", "rewards", "masks", "bad_masks", "active_masks"):
            dst, src = getattr(shared_buffer, name, None), views[name]
            if dst is None or src is None:
                continue
            if tuple(dst.shape) != tuple(src.shape):
                raise ValueError("SharedReplayBuffer.%s is %s, this rollout gives %s" % (name, tuple(dst.shape), tuple(src.shape)))
            dst.copy_(src)
        shared_buffer.step = 0
        return shared_buffer


class PolicyRollout:
    """T-step on-device rollout of one env handle under one ``FusedPolicy`` handle.

    ``tile_policy`` (int32 ``[ceil(P*N/128)]``, device) selects the (actor, critic) weight set per
    tile of 128 agent rows; rows are seat-major (row = seat*N + world).  ``None`` = set 0 for
    everybody (plain self-play, train/trainer.py:41-44)."""

    def __init__(self, env: B200Overcooked, policy: FusedPolicy, T: int, tile_policy: Optional[torch.Tensor] = None,
                 with_critic: bool = True, with_logp: bool = True, seed: int = 0, use_graph: bool = False,
                 fused: Optional[bool] = None, policy_index: int = 0, world_offset: int = 0,
                 total_worlds: Optional[int] = None, critic_policy: Optional[torch.Tensor] = None,
                 weights: Optional[Sequence] = None):
        """``total_worlds`` (with ``world_offset`` = global index of this env's world 0): key the action sampling by
        the GLOBAL (seat, world) so that a sharded run draws exactly the streams of the unsharded one
        (``ocb_policy_set_sampling_rows``); ``None`` keeps the launch-local rows.

        ``fused``: run the rollout as ONE persistent launch (``ocb_rollout_policy_fused``: self-play of weight
        set ``policy_index``, hidden 64, critic on); ``None`` = use it whenever it applies, ``False`` = always the
        2T+1-launch path.  Both paths fill bit-identical buffers.  A ``tile_policy`` whose two seat halves are equal
        (``pair_tile_policy([(p0, p0), (p1, p1), ...], worlds_per_slice)``) with the critic on is population self-play:
        it runs as one launch too (``ocb_rollout_population_fused``).  The table is classified once, here: the launches
        read the caller's tensor, so in-place edits take effect (also in graph replays) but must keep the two halves
        equal; build a new ``PolicyRollout`` for a table that mixes policies across seats.

        ``critic_policy`` (int32 ``[2N/128]``, the seat tiles of ``tile_policy``; needs ``tile_policy`` and ``with_critic``):
        cross-play TRAINING collection, XD's SP / XP slices.  Seat tile k acts with ``tile_policy[k]``'s actor and is valued
        by ``critic_policy[k]``'s critic, or not at all for -1 (a partner's seat): its ``value_preds`` slots stay 0.0.
        ``crossplay_training_tables`` builds both tables.  ``fused=None`` runs the cross-play launch plus one critic pass
        (``ocb_rollout_crossplay_train_fused``), falling back to per-step actor launches and per-step critic passes where
        that is unsupported (hidden 512, layouts outside the fused kernel); ``fused=True`` raises ``NativeError`` there.
        Both tables are checked once, here (entries -1 or below ``n_policies``; ``tile_policy`` entries 0 or more); the
        launches read the caller's tensors.

        ``weights``: ``(index, actor, critic)`` sets as ``FusedPolicy.set_weights_device`` takes them.  Every ``collect()``
        then first packs their current values into the handle on the device, in the same stream as the collection; with
        ``use_graph`` the refresh is part of the captured graph, so one replay loads the parameters the nets hold at that
        moment (nets made with ``PolicyNet.alias_state_dict`` follow the trainer's optimizer) and collects with them."""
        if env.num_players != policy.layout.num_players:
            raise ValueError("env and policy were built for different player counts")
        if env.sim_device != policy.device:
            raise ValueError("env and policy live on different devices")
        if (policy.layout.width, policy.layout.height) != (env.width, env.height):
            raise ValueError("env and policy were built for different layouts")
        M = env.num_players * env.num_envs
        if tile_policy is not None:
            if tile_policy.dtype != torch.int32 or tile_policy.numel() != (M + TILE - 1) // TILE:
                raise ValueError("tile_policy must be int32 [%d]" % ((M + TILE - 1) // TILE))
            tile_policy = tile_policy.to(env.sim_device).contiguous()
        if critic_policy is not None:
            if tile_policy is None or not with_critic:
                raise ValueError("critic_policy needs tile_policy and with_critic=True")
            if env.num_envs % TILE != 0:
                raise ValueError("critic_policy needs a multiple of %d worlds (one critic per 128-row seat tile)" % TILE)
            if critic_policy.dtype != torch.int32 or critic_policy.numel() != tile_policy.numel():
                raise ValueError("critic_policy must be int32 [%d]" % tile_policy.numel())
            critic_policy = critic_policy.to(env.sim_device).contiguous()
            for name, table, low in (("tile_policy", tile_policy, 0), ("critic_policy", critic_policy, -1)):
                host = table.cpu()
                if bool(((host < low) | (host >= policy.n_policies)).any()):
                    raise ValueError("%s entries must lie in [%d, %d)" % (name, low, policy.n_policies))
        self.weights = None
        if weights is not None:
            self.weights = list(weights)
            policy._weight_srcs(self.weights)  # shape / dtype / device errors now rather than at the first collect
        self.env, self.policy, self.T, self.seed = env, policy, T, seed
        self.tile_policy, self.critic_policy = tile_policy, critic_policy
        self.buf = RolloutBuffer(env, T, with_critic, with_logp)
        self._lib = _native.lib()
        self.policy_index = policy_index
        # one persistent launch needs the tensor-core policy path: 2 players, grids up to 6 rows (else per-step launches,
        # which run any shape — the generic policy kernel covers schelling / corridor / multiplayer_schelling ...)
        # (self-play of one policy with its critic, or cross-play slices without a critic: ocb_rollout_crossplay_fused,
        # or self-play slices of a population with their critics: ocb_rollout_population_fused)
        small = policy.hidden == 64 and env.num_players == 2
        self._slice_policy = None
        if critic_policy is not None:
            # slots of -1 tiles are never written by the fused path; the per-step fallback zeroes them after its critic pass
            self.buf.value_preds.zero_()
            self._no_value = (critic_policy < 0).view(1, -1, 1)
            self._critic_filled = critic_policy.clamp(min=0)  # -1 -> weight set 0, whose values are then zeroed
            self.fused = small if fused is None else bool(fused)
            self._fused_required = bool(fused)
        elif tile_policy is not None and with_critic and env.num_players == 2 and env.num_envs % TILE == 0:
            half = tile_policy.numel() // 2
            host = tile_policy.cpu()
            if torch.equal(host[:half], host[half:]):
                self._slice_policy = tile_policy[:half]
        population = self._slice_policy is not None
        can_fuse = small and ((tile_policy is None and with_critic) or population or
                              (tile_policy is not None and not with_critic and env.num_envs % TILE == 0))
        if fused and population and not small:
            raise _native.NativeError(_native.OCB_ERR_UNSUPPORTED, "the population launch exists for hidden_size 64 only")
        # fused=True on a population table of a layout the fused kernel does not take (generic-kernel layouts, layouts too
        # large for its shared memory) is answered by the launch itself: OCB_ERR_UNSUPPORTED, raised at collect()
        # (so is fused=True with a critic_policy: hidden 512 included)
        if fused and not (can_fuse or population or critic_policy is not None):
            raise ValueError("the fused rollout needs hidden 64, two players and either self-play of one policy with its critic "
                             "or cross-play slices (tile_policy, a multiple of %d worlds) without one" % TILE)
        if critic_policy is None:
            self.fused = can_fuse if fused is None else bool(fused)
            self._fused_required = bool(fused)
        if tile_policy is None and policy_index != 0 and not self.fused:
            self.tile_policy = tile_policy = torch.full(((M + TILE - 1) // TILE,), policy_index, dtype=torch.int32,
                                                        device=env.sim_device)
        self._primed = False
        self._graphs = {}
        self.use_graph = use_graph
        self.rollouts = 0
        N = env.num_envs
        if total_worlds is not None and not (0 <= world_offset and world_offset + N <= total_worlds):
            raise ValueError("world_offset + num_envs must lie inside total_worlds")
        self._sampling_rows = (0, 0, 0) if total_worlds is None else (N, world_offset, total_worlds - N + world_offset)

    # ------------------------------------------------------------------ launches
    def _issue(self, deterministic: bool):
        b, env = self.buf, self.env
        stream = ctypes.c_void_p(torch.cuda.current_stream(env.sim_device).cuda_stream)
        # handle-level state, set per issue: several rollouts may share one policy handle
        _native.check(self._lib.ocb_policy_set_sampling_rows(self.policy._h, *self._sampling_rows))
        if self.weights is not None:
            self.policy.set_weights_device(self.weights)
        if self.fused:
            if self.critic_policy is not None:
                rc = self._lib.ocb_rollout_crossplay_train_fused(
                    env._h, self.policy._h, self.T, _ptr(self.tile_policy), _ptr(self.critic_policy), _ptr(b.obs),
                    _ptr(b.actions), _ptr(b.action_log_probs), _ptr(b.value_preds), _ptr(b.rewards), _ptr(b.dones),
                    int(deterministic), self.seed, stream)
            elif self._slice_policy is not None:
                rc = self._lib.ocb_rollout_population_fused(
                    env._h, self.policy._h, self.T, _ptr(self._slice_policy), _ptr(b.obs), _ptr(b.actions),
                    _ptr(b.action_log_probs), _ptr(b.value_preds), _ptr(b.rewards), _ptr(b.dones), int(deterministic),
                    self.seed, stream)
            elif self.tile_policy is not None:
                rc = self._lib.ocb_rollout_crossplay_fused(
                    env._h, self.policy._h, self.T, _ptr(self.tile_policy), _ptr(b.obs), _ptr(b.actions),
                    _ptr(b.action_log_probs), _ptr(b.rewards), _ptr(b.dones), int(deterministic), self.seed, stream)
            else:
                rc = self._lib.ocb_rollout_policy_fused(
                    env._h, self.policy._h, self.T, self.policy_index, _ptr(b.obs), _ptr(b.actions), _ptr(b.action_log_probs),
                    _ptr(b.value_preds), _ptr(b.rewards), _ptr(b.dones), int(deterministic), self.seed, stream)
            if rc != _native.OCB_ERR_UNSUPPORTED or self._fused_required:
                _native.check(rc)
                return
            self.fused = False  # layout too large for the fused kernel: per-step launches from here on
        if self.critic_policy is not None:
            self._issue_crossplay_train_steps(deterministic, stream)
            return
        _native.check(self._lib.ocb_rollout_policy(
            env._h, self.policy._h, self.T, _ptr(self.tile_policy), _ptr(b.obs), _ptr(b.actions),
            _ptr(b.action_log_probs), _ptr(b.value_preds), _ptr(b.rewards), _ptr(b.dones), int(deterministic),
            self.seed, stream))

    def _issue_crossplay_train_steps(self, deterministic: bool, stream):
        """the per-step form of ocb_rollout_crossplay_train_fused: the actors through ocb_rollout_policy without a critic, then
        one critic pass per step (a single pass over all T + 1 steps would size the hidden-512 activation scratch for the
        whole slab), then the slots of -1 tiles zeroed"""
        b, env, M = self.buf, self.env, self.env.num_players * self.env.num_envs
        _native.check(self._lib.ocb_rollout_policy(
            env._h, self.policy._h, self.T, _ptr(self.tile_policy), _ptr(b.obs), _ptr(b.actions), _ptr(b.action_log_probs),
            None, _ptr(b.rewards), _ptr(b.dones), int(deterministic), self.seed, stream))
        for t in range(self.T + 1):
            _native.check(self._lib.ocb_policy_value(self.policy._h, _ptr(b.obs[t]), M, _ptr(self._critic_filled),
                                                     _ptr(b.value_preds[t]), stream))
        b.value_preds.view(self.T + 1, -1, TILE).masked_fill_(self._no_value, 0.0)

    def prime(self):
        """slot 0 <- observation of the env's CURRENT state.  Always re-observed (one cheap launch): the env may have
        moved between two rollouts (``n_reset``, ``set_state``, another ``n_step`` / rollout on the same handle), and
        copying the previous rollout's last slot (SharedReplayBuffer.after_update, shared_buffer.py:222-226) would then
        pair a stale obs[0] with actions and values computed from the new state.  When nothing moved the result is the
        same bytes as that copy."""
        with torch.cuda.device(self.env.sim_device):
            _native.check(self._lib.ocb_observe(self.env._h, _ptr(self.buf.obs[0]), self.env._stream()))
            self._primed = True

    def collect(self, deterministic: bool = False) -> RolloutBuffer:
        """One T-step rollout, asynchronous on torch's current stream."""
        with torch.cuda.device(self.env.sim_device):
            self.prime()
            if not self.use_graph:
                self._issue(deterministic)
            else:
                g = self._graphs.get(bool(deterministic))
                if g is None:
                    g = self._capture(deterministic)
                g.replay()
        self.rollouts += 1
        return self.buf

    def _capture(self, deterministic: bool):
        """capture the 2T+1 launches once; replays read the sampling offset from the device step
        counter, so they draw fresh actions"""
        _native.check(self._lib.ocb_policy_reserve(self.policy._h, self.env.num_players * self.env.num_envs))
        torch.cuda.synchronize(self.env.sim_device)
        # capture does not execute: the env state is untouched, only the launch sequence is recorded
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            self._issue(deterministic)
        self._graphs[bool(deterministic)] = g
        return g

    # ------------------------------------------------------------------ scores
    def episode_stats(self):
        return self.env.episode_stats()

    def mean_episode_return(self) -> float:
        rs, ep = self.env.episode_stats()
        n = int(ep.sum().item())
        return float(rs.sum().item()) / n if n else float("nan")

    def slice_episode_returns(self, worlds_per_slice: int):
        """(sum of episode returns int64 [S], episodes int64 [S]) per contiguous slice of ``worlds_per_slice`` worlds, on
        the device: the per-member scores of a population trained on self-play slices (as ``CrossPlayEvaluator.run``)"""
        N = self.env.num_envs
        if worlds_per_slice <= 0 or N % worlds_per_slice != 0:
            raise ValueError("worlds_per_slice must divide the env's %d worlds" % N)
        rs, ep = self.env.episode_stats()
        n = N // worlds_per_slice
        return rs.view(n, worlds_per_slice).sum(1), ep.view(n, worlds_per_slice).sum(1, dtype=torch.int64)


# ---------------------------------------------------------------------------- cross-play
def crossplay_training_tables(slices: Sequence, worlds_per_slice: int, device=None):
    """(tile_policy, critic_policy) of a cross-play training collection (``PolicyRollout(..., critic_policy=...)``): the env's
    worlds are ``len(slices)`` contiguous slices of ``worlds_per_slice`` worlds, slice s given as ``((actor0, critic0),
    (actor1, critic1))`` weight-set indices per seat; a critic of ``None`` (a seat whose values are not needed) becomes -1.

    XD (train/XD/xd_player.py:177-230), the ego ``e`` with SP / XP critics ``sp``, ``xp0[j]``, ``xp1[j]`` against partners
    ``p[j]``: ``[((e, sp), (e, sp))] + [((e, xp0[j]), (p[j], None)) for j] + [((p[j], None), (e, xp1[j])) for j]``.  Best
    response (train/MultiConvention/xd_player.py:66-171): ``[((e, e), (p[j], None)) for j] + [((p[j], None), (e, e)) for j]``."""
    sl = [tuple(tuple(seat) for seat in s) for s in slices]
    if not sl or any(len(s) != 2 or any(len(seat) != 2 for seat in s) for s in sl):
        raise ValueError("each slice is ((actor0, critic0), (actor1, critic1))")
    actors = pair_tile_policy([(s[0][0], s[1][0]) for s in sl], worlds_per_slice, device)
    critics = pair_tile_policy([tuple(-1 if seat[1] is None else seat[1] for seat in s) for s in sl], worlds_per_slice, device)
    return actors, critics


def pair_tile_policy(pairs: Sequence[Sequence[int]], worlds_per_pair: int, device=None) -> torch.Tensor:
    """tile_policy of an env whose worlds are ``len(pairs)`` contiguous slices of ``worlds_per_pair``
    worlds, slice s played by (seat 0: policy pairs[s][0], seat 1: policy pairs[s][1]) — the layout of
    XDPlayer / CentralizedMultiAgent (xd_player.py:190-207, partner_agents.py:97-111) generalised to
    arbitrary pairs.  Rows are seat-major, so the table is [seat-0 tiles..., seat-1 tiles...]."""
    if worlds_per_pair % TILE != 0:
        raise ValueError("worlds_per_pair must be a multiple of %d (one weight set per 128-row tile)" % TILE)
    tiles_per_pair = worlds_per_pair // TILE
    p = torch.as_tensor(list(pairs), dtype=torch.int32).reshape(-1, 2)
    table = torch.cat([p[:, 0].repeat_interleave(tiles_per_pair), p[:, 1].repeat_interleave(tiles_per_pair)])
    return table.to(device) if device is not None else table


class CrossPlayEvaluator:
    """Cross-play return matrix of a population (BASELINE config 5; the all-pairs generalisation of
    the xp_scores of train/XD/xd_player.py:143-149 and of train/testing.py:39-59).

    This rank evaluates ``pairs`` (a list of (i, j) policy indices): one env with
    ``len(pairs) * worlds_per_pair`` worlds, actors only, one episode of ``horizon`` steps per world.
    ``run()`` returns per-pair (sum of episode returns, number of episodes) on the device;
    ``sharding.gather_pair_matrix`` assembles the [n, n] matrix across ranks."""

    def __init__(self, layout: str, policy: FusedPolicy, pairs, worlds_per_pair: int = 1024, horizon: int = 400,
                 gpu_id: int = 0, seed: int = 0, world_offset: int = 0, chunk_steps: int = 50, use_graph: bool = True,
                 deterministic: bool = False, total_worlds: Optional[int] = None, fused: Optional[bool] = None):
        self.pairs = [tuple(int(v) for v in p) for p in pairs]
        if not self.pairs:
            raise ValueError("no pairs on this rank")
        if max(max(p) for p in self.pairs) >= policy.n_policies:
            raise ValueError("pair refers to a policy the handle does not hold")
        if horizon % chunk_steps != 0:
            raise ValueError("horizon must be a multiple of chunk_steps")
        self.worlds_per_pair, self.horizon, self.chunk_steps = worlds_per_pair, horizon, chunk_steps
        self.deterministic = deterministic
        N = len(self.pairs) * worlds_per_pair
        self.env = B200Overcooked(layout, N, gpu_id, horizon=horizon, seed=seed, world_offset=world_offset)
        table = pair_tile_policy(self.pairs, worlds_per_pair, self.env.sim_device)
        self.table, self.policy, self.seed = table, policy, seed
        self._sampling_rows = (0, 0, 0) if total_worlds is None else (N, world_offset, total_worlds - N + world_offset)
        # The whole episode as ONE persistent launch without any trajectory buffer (ocb_rollout_crossplay_fused) when the
        # fused kernel takes the shape; ``fused=False`` (or a layout it does not fit) runs chunked per-step launches.
        self.fused = (fused if fused is not None else True) and policy.hidden == 64 and self.env.num_players == 2 and N % TILE == 0
        # the slab holds chunk_steps observations, not the whole episode: evaluation keeps no trajectory
        # total_worlds = worlds of the whole pair list over all ranks: the matrix then does not depend on the sharding
        self._rollout_args = dict(T=chunk_steps, tile_policy=table, with_critic=False, with_logp=False, seed=seed,
                                  use_graph=use_graph, fused=False, world_offset=world_offset, total_worlds=total_worlds)
        # the chunked per-step rollout (and its observation slab) is only built when it is needed
        self.rollout = None if self.fused else PolicyRollout(self.env, policy, **self._rollout_args)

    def _run_fused(self) -> bool:
        lib, env = _native.lib(), self.env
        with torch.cuda.device(env.sim_device):
            stream = ctypes.c_void_p(torch.cuda.current_stream(env.sim_device).cuda_stream)
            _native.check(lib.ocb_policy_set_sampling_rows(self.policy._h, *self._sampling_rows))
            rc = lib.ocb_rollout_crossplay_fused(env._h, self.policy._h, self.horizon, _ptr(self.table), None, None, None, None,
                                                 None, int(self.deterministic), self.seed, stream)
        if rc == _native.OCB_ERR_UNSUPPORTED:
            return False
        _native.check(rc)
        return True

    def run(self):
        """one full episode per world -> (return_sum int64 [pairs], episodes int64 [pairs]) on the device"""
        self.env.n_reset()
        self.env.clear_episode_stats()
        if self.fused and not self._run_fused():
            self.fused = False
        if not self.fused:
            if self.rollout is None:
                self.rollout = PolicyRollout(self.env, self.policy, **self._rollout_args)
            self.rollout._primed = False
            for _ in range(self.horizon // self.chunk_steps):
                self.rollout.collect(self.deterministic)
        rs, ep = self.env.episode_stats()
        n = len(self.pairs)
        return rs.view(n, self.worlds_per_pair).sum(1), ep.view(n, self.worlds_per_pair).sum(1, dtype=torch.int64)

    def close(self):
        self.env.close()
