"""Mixed-play ("MP") data collection on the device (``ocb_rollout_mixed_fused``, csrc/rollout_fused.cuh, or the per-step
``ocb_rollout_mixed``, csrc/mixed_kernels.cu).

Replaces, for the CoMeDi / XD trainer of the reference:

* ``XDPlayer.collect_mp_episode`` / ``next_mp_step`` (train/XD/xd_player.py:232-356): 2L env steps over
  ``envs_mp`` (G = L - 1 worlds, train/XD/serial.py:29), the ego seat's per-world random switch between the
  policy being trained and the partner convention, and the growing block of worlds that is forced back to the
  trained policy;
* ``MixedAgent.get_action`` / ``update`` (train/partner_agents.py:151-244): the same for the partner seat;
* ``SharedReplayBuffer.diaginsert`` / ``partinsert`` (train/MAPPO/utils/shared_buffer.py:150-220): a dozen strided
  torch copies per step that put the forced worlds on a diagonal / a row prefix of the buffer.

Here one env holds ``replicas`` independent copies of the G-world scheme and nothing synchronises.  A collection is one
persistent launch of the fused rollout kernel plus one critic launch over the recorded observations (hidden 64, the layouts
the tensor-core kernels take), else ``10 L + 4`` per-step launches; both issued from C (or one CUDA-graph launch), both
filling the same buffers bit for bit.  The buffer is seat-major
(``[L(+1), P, N, ...]``, int8 observations); ``shared_buffer_views()`` gives the reference's ``[L(+1), N, P, ...]``
axis order as zero-copy views.
"""
from __future__ import annotations

import ctypes
from typing import Dict, Optional, Sequence

import torch

from . import _native
from .overcooked_env import B200Overcooked, _ptr
from .policy import FusedPolicy


class MixedPlayBuffer:
    """``mp_buf`` of the reference (generate_buffer(args, env_mp, device, env_length - 1), train/XD/serial.py:43),
    seat-major on the device.  ``dones[t]`` is stored at the SAME slot as the observation (diaginsert / partinsert
    store ``masks = 1 - done`` at slot t, chooseinsert at t + 1)."""

    def __init__(self, env: B200Overcooked, L: int):
        P, N, dev = env.num_players, env.num_envs, env.sim_device
        self.L, self.P, self.N = L, P, N
        self.obs = torch.zeros((L + 1, P, N, env.width, env.height, env.channels), dtype=torch.int8, device=dev)
        self.actions = torch.zeros((L, P, N), dtype=torch.int32, device=dev)
        self.action_log_probs = torch.zeros((L, P, N), dtype=torch.float32, device=dev)
        self.value_preds = torch.zeros((L + 1, P, N), dtype=torch.float32, device=dev)
        self.rewards = torch.zeros((L, P, N), dtype=torch.int32, device=dev)
        self.dones = torch.zeros((L, N), dtype=torch.int32, device=dev)

    def dones_for_returns(self) -> torch.Tensor:
        """``compute_returns`` multiplies step t by ``masks[t+1]`` (shared_buffer.py:262-275); with the masks of this
        buffer stored at their own slot that is ``1 - dones[t+1]`` for t < L-1 and the never-written
        ``masks[L] = 1`` for the last step -> the ``done [L,N]`` input of ``ocb_compute_returns``."""
        d = torch.zeros_like(self.dones)
        d[:-1] = self.dones[1:]
        return d

    def compute_returns(self, gamma: float = 0.99, gae_lambda: float = 0.95, use_gae: bool = True, value_normalizer=None,
                        normalize: bool = True):
        from .returns import compute_returns
        self.returns, self.advantages = compute_returns(
            self.value_preds, self.rewards, self.dones_for_returns(), gamma, gae_lambda, use_gae, value_normalizer,
            normalize, getattr(self, "returns", None), getattr(self, "advantages", None))
        return self.returns, self.advantages

    def shared_buffer_views(self) -> Dict[str, torch.Tensor]:
        """zero-copy views with the reference's names and ``[L(+1), N, P, ...]`` axis order; ``masks`` is
        materialised (``[L+1, N, P, 1]`` float, slot L = 1)."""
        sw = lambda t: t.transpose(1, 2)
        obs = sw(self.obs)
        masks = torch.ones((self.L + 1, self.N, self.P, 1), dtype=torch.float32, device=self.obs.device)
        masks[:-1] = (1 - self.dones).to(torch.float32)[:, :, None, None]
        return {"obs": obs, "share_obs": obs, "actions": sw(self.actions).unsqueeze(-1),
                "action_log_probs": sw(self.action_log_probs).unsqueeze(-1),
                "value_preds": sw(self.value_preds).unsqueeze(-1), "rewards": sw(self.rewards).unsqueeze(-1),
                "masks": masks}


class MixedPlayCollector:
    """One mixed-play collection = 2L env steps of an env with ``replicas * (L - 1)`` worlds.

    ``policy`` holds the weight sets: ``main_policy`` = (actor being trained, its mixed-play critic ``mp_critic``,
    train/XD/MCPolicy.py:21,60), ``partner_policy`` = the partner convention (only its actor is used).  The env is
    not reset: like the reference the collection continues from the env's current state.

    ``fused``: ``None`` runs the collection as one persistent launch (``ocb_rollout_mixed_fused``) whenever it applies and
    falls back to the per-step launches for good when the library answers ``OCB_ERR_UNSUPPORTED`` (hidden 512, layouts
    outside the tensor-core kernels or too large for the fused kernel); ``True`` raises ``NativeError`` there instead;
    ``False`` always runs the per-step path.  ``.fused`` tells which path ran.

    ``weights``: ``(index, actor, critic)`` sets as ``FusedPolicy.set_weights_device`` takes them, refreshed on the device at
    the start of every ``collect()`` (inside the captured graph with ``use_graph``), as for ``PolicyRollout``.  Slot L of
    ``value_preds`` is main's critic on the all-zero observation as the handle holds it when the collection runs."""

    def __init__(self, env: B200Overcooked, policy: FusedPolicy, L: int, main_policy: int = 0, partner_policy: int = 1,
                 seed: int = 0, mix_seed: int = 0, use_graph: bool = False, fused: Optional[bool] = None,
                 weights: Optional[Sequence] = None):
        if env.num_players != 2:
            raise ValueError("mixed play supports 2 players")
        if env.sim_device != policy.device:
            raise ValueError("env and policy live on different devices")
        if (policy.layout.width, policy.layout.height) != (env.width, env.height):
            raise ValueError("env and policy were built for different layouts")
        if L < 2 or env.num_envs % (L - 1) != 0:
            raise ValueError("the env must hold a multiple of L - 1 = %d worlds (envs_mp of the reference has "
                             "exactly L - 1)" % (L - 1))
        if not (0 <= main_policy < policy.n_policies and 0 <= partner_policy < policy.n_policies):
            raise ValueError("policy index out of range")
        self.weights = None
        if weights is not None:
            self.weights = list(weights)
            policy._weight_srcs(self.weights)  # shape / dtype / device errors now rather than at the first collect
        self.env, self.policy, self.L = env, policy, L
        self.main_policy, self.partner_policy = main_policy, partner_policy
        self.seed, self.mix_seed = seed, mix_seed
        self.replicas = env.num_envs // (L - 1)
        self.buf = MixedPlayBuffer(env, L)
        self._lib = _native.lib()
        self.fused = policy.hidden == 64 if fused is None else bool(fused)
        self._fused_required = bool(fused)
        self._scratch = None if fused else self._alloc_scratch()  # the per-step path's turn data, where that path can run
        self.use_graph = use_graph
        self._graph = None
        self.collections = 0

    def _alloc_scratch(self) -> torch.Tensor:
        nbytes = int(self._lib.ocb_rollout_mixed_scratch_bytes(self.env._h))
        return torch.empty((nbytes,), dtype=torch.uint8, device=self.env.sim_device)

    def _issue(self, deterministic: bool):
        b, env = self.buf, self.env
        stream = ctypes.c_void_p(torch.cuda.current_stream(env.sim_device).cuda_stream)
        # launch-local sampling rows (a sharded PolicyRollout may have left global rows on a shared policy handle)
        _native.check(self._lib.ocb_policy_set_sampling_rows(self.policy._h, 0, 0, 0))
        if self.weights is not None:
            self.policy.set_weights_device(self.weights)
        if self.fused:
            rc = self._lib.ocb_rollout_mixed_fused(
                env._h, self.policy._h, self.L, self.main_policy, self.partner_policy, _ptr(b.obs), _ptr(b.actions),
                _ptr(b.action_log_probs), _ptr(b.value_preds), _ptr(b.rewards), _ptr(b.dones), int(deterministic),
                self.seed, self.mix_seed, stream)
            if rc != _native.OCB_ERR_UNSUPPORTED or self._fused_required:
                _native.check(rc)
                return
            self.fused = False  # the library launched nothing: per-step launches from here on
        _native.check(self._lib.ocb_rollout_mixed(
            env._h, self.policy._h, self.L, self.main_policy, self.partner_policy, _ptr(b.obs), _ptr(b.actions),
            _ptr(b.action_log_probs), _ptr(b.value_preds), _ptr(b.rewards), _ptr(b.dones), int(deterministic), self.seed,
            self.mix_seed, _ptr(self._scratch), self._scratch.numel(), stream))

    def collect(self, deterministic: bool = False) -> MixedPlayBuffer:
        """asynchronous on torch's current stream"""
        with torch.cuda.device(self.env.sim_device):
            if not self.use_graph:
                self._issue(deterministic)
            else:
                if self._graph is None or self._graph[0] != bool(deterministic):
                    _native.check(self._lib.ocb_policy_reserve(self.policy._h, self.env.num_players * self.env.num_envs))
                    torch.cuda.synchronize(self.env.sim_device)
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g):  # capture records the launches, the env state is untouched
                        self._issue(deterministic)
                    self._graph = (bool(deterministic), g)
                self._graph[1].replay()
        self.collections += 1
        return self.buf

    def mp_scores(self):
        """(sum of episode returns, episodes) per world, as accumulated on the device (mp_scores /
        running_mp_score of xd_player.py:352-356)"""
        return self.env.episode_stats()
