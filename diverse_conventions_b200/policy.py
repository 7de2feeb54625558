"""MAPPO actor / critic networks of the reference, as weight containers for the fused
sm_100a forward kernel plus a plain PyTorch fp32 forward used as the numerical reference.

Reference architecture (CNN branch, taken because the observation is 3-D):
``R_Actor`` / ``R_Critic`` train/MAPPO/r_actor_critic.py:12-71,142-197, ``CNNLayer``
train/MAPPO/utils/cnn.py:11-42 (``x.movedim(-1,-3)`` -> Conv2d(C -> h/2, k=3, s=1, no pad) ->
ReLU -> flatten -> Linear((h/2)(W-2)(H-2) -> h) -> ReLU -> Linear(h -> h) -> ReLU), action
head ``Categorical`` train/MAPPO/utils/distributions.py:55-68 (Linear(h -> 6), orthogonal
gain 0.01), value head ``v_out`` Linear(h -> 1).  State-dict keys are the reference's
(SURVEY.md appendix B.18), so checkpoints load either way:
    actor : base.cnn.cnn.{0,3,5}.{weight,bias}, act.action_out.linear.{weight,bias}
    critic: base.cnn.cnn.{0,3,5}.{weight,bias}, v_out.{weight,bias}
"""
from __future__ import annotations

import math
from typing import Dict

import torch
import torch.nn.functional as F

NUM_ACTIONS = 6
_BASE_KEYS = ("base.cnn.cnn.0", "base.cnn.cnn.3", "base.cnn.cnn.5")
_WEIGHTS = ("conv_w", "conv_b", "fc1_w", "fc1_b", "fc2_w", "fc2_b", "head_w", "head_b")  # in state_dict() order


class PolicyNet:
    """One network (actor or critic).  Tensors are fp32 and live on `device`."""

    def __init__(self, kind: str, width: int, height: int, channels: int, hidden: int, device="cpu"):
        assert kind in ("actor", "critic")
        self.kind, self.W, self.H, self.C, self.hidden = kind, width, height, channels, hidden
        self.conv_out = hidden // 2
        self.npos = (width - 2) * (height - 2)
        self.head_key = "act.action_out.linear" if kind == "actor" else "v_out"
        self.head_out = NUM_ACTIONS if kind == "actor" else 1
        self.device = torch.device(device)
        z = lambda *s: torch.zeros(*s, dtype=torch.float32, device=self.device)
        self.conv_w, self.conv_b = z(self.conv_out, channels, 3, 3), z(self.conv_out)
        self.fc1_w, self.fc1_b = z(hidden, self.conv_out * self.npos), z(hidden)
        self.fc2_w, self.fc2_b = z(hidden, hidden), z(hidden)
        self.head_w, self.head_b = z(self.head_out, hidden), z(self.head_out)

    # ------------------------------------------------------------------ weights
    def init_like_reference(self, seed: int, gain: float = 0.01) -> "PolicyNet":
        """orthogonal init, relu gain for the base, `gain` for the action head, gain 1 for v_out,
        zero biases (train/MAPPO/utils/util.py:14-17, cnn.py:15-20, distributions.py:58-62,
        r_actor_critic.py:168-174).  Not bit-identical to the reference's RNG consumption."""
        g = torch.Generator().manual_seed(seed)
        relu_gain = math.sqrt(2.0)

        def ortho(shape, gn):
            w = torch.empty(shape)
            rows, cols = shape[0], int(torch.tensor(shape[1:]).prod())
            a = torch.randn((max(rows, cols), min(rows, cols)), generator=g)
            q, r = torch.linalg.qr(a)
            q = q * torch.sign(torch.diagonal(r))
            if rows < cols:
                q = q.t()
            w.copy_((gn * q[:rows, :cols]).reshape(shape))
            return w.to(self.device)

        self.conv_w = ortho(tuple(self.conv_w.shape), relu_gain)
        self.fc1_w = ortho(tuple(self.fc1_w.shape), relu_gain)
        self.fc2_w = ortho(tuple(self.fc2_w.shape), relu_gain)
        self.head_w = ortho(tuple(self.head_w.shape), gain if self.kind == "actor" else 1.0)
        for b in (self.conv_b, self.fc1_b, self.fc2_b, self.head_b):
            b.zero_()
        return self

    def state_dict(self) -> Dict[str, torch.Tensor]:
        k0, k3, k5 = _BASE_KEYS
        return {k0 + ".weight": self.conv_w, k0 + ".bias": self.conv_b, k3 + ".weight": self.fc1_w,
                k3 + ".bias": self.fc1_b, k5 + ".weight": self.fc2_w, k5 + ".bias": self.fc2_b,
                self.head_key + ".weight": self.head_w, self.head_key + ".bias": self.head_b}

    def load_state_dict(self, sd) -> "PolicyNet":
        mine = self.state_dict()
        missing = [k for k in mine if k not in sd]
        if missing:
            raise KeyError("state dict lacks %s" % missing)
        for k, dst in mine.items():
            src = torch.as_tensor(sd[k], dtype=torch.float32)
            if tuple(src.shape) != tuple(dst.shape):
                raise ValueError("%s: shape %s, expected %s" % (k, tuple(src.shape), tuple(dst.shape)))
            dst.copy_(src)
        return self

    def alias_state_dict(self, sd) -> "PolicyNet":
        """Like ``load_state_dict``, but the net keeps references to the given tensors instead of copying them.  A net
        built from ``module.state_dict()`` of the reference's ``R_Actor`` / ``R_Critic`` therefore sees the optimizer's
        in-place updates, and ``FusedPolicy.set_weights_device`` (or a collector given ``weights=``) packs the current
        values.  Each tensor must have its shape, be fp32 and contiguous, and live on this net's device (``ValueError``)."""
        mine = self.state_dict()
        missing = [k for k in mine if k not in sd]
        if missing:
            raise KeyError("state dict lacks %s" % missing)
        want = self.device
        if want.type == "cuda" and want.index is None:
            want = torch.device("cuda", torch.cuda.current_device())
        keep = []
        for k, dst in mine.items():
            src = sd[k]
            if not isinstance(src, torch.Tensor):
                raise ValueError("%s: expected a tensor, got %s" % (k, type(src).__name__))
            if tuple(src.shape) != tuple(dst.shape):
                raise ValueError("%s: shape %s, expected %s" % (k, tuple(src.shape), tuple(dst.shape)))
            if src.dtype != torch.float32:
                raise ValueError("%s: dtype %s, expected torch.float32" % (k, src.dtype))
            if not src.is_contiguous():
                raise ValueError("%s is not contiguous" % k)
            if src.device != want:
                raise ValueError("%s lives on %s, this net on %s" % (k, src.device, want))
            keep.append(src.detach())
        for name, t in zip(_WEIGHTS, keep):
            setattr(self, name, t)
        return self

    # ------------------------------------------------------------------ fp32 reference forward
    @torch.no_grad()
    def features(self, obs: torch.Tensor) -> torch.Tensor:
        x = obs.to(self.device, torch.float32).movedim(-1, -3)  # (M, C, W, H), cnn.py:41
        x = F.relu(F.conv2d(x, self.conv_w, self.conv_b)).flatten(1)
        x = F.relu(F.linear(x, self.fc1_w, self.fc1_b))
        return F.relu(F.linear(x, self.fc2_w, self.fc2_b))

    @torch.no_grad()
    def forward(self, obs: torch.Tensor) -> torch.Tensor:
        """actor: logits [M, 6] (== R_Actor.get_logits(...).logits before normalisation, all actions
        available); critic: values [M, 1] (R_Critic.forward)."""
        return F.linear(self.features(obs), self.head_w, self.head_b)


def log_softmax_sample(logits: torch.Tensor, actions: torch.Tensor) -> torch.Tensor:
    """log pi(a) as FixedCategorical.log_probs computes it (distributions.py:14-25)."""
    return torch.log_softmax(logits, dim=-1).gather(-1, actions.long().reshape(-1, 1)).squeeze(-1)


class FusedPolicy:
    """Device handle of the fused tensor-core forward (ocb_policy_*, csrc/policy_kernels.cu).

    Holds `n_policies` (actor, critic) weight sets for one layout; rows are processed in tiles of
    128 and `tile_policy` picks the weight set per tile (cross-play slices)."""

    TILE = 128

    def __init__(self, layout_params, hidden: int = 64, n_policies: int = 1, gpu_id: int = 0):
        import ctypes
        from . import _native
        if not torch.cuda.is_available():
            raise RuntimeError("FusedPolicy needs a CUDA device; there is no CPU fallback")
        self._ct, self._native = ctypes, _native
        self._lib = _native.lib()
        self.layout = layout_params
        self.hidden, self.n_policies = hidden, n_policies
        self.device = torch.device("cuda", gpu_id)
        self._cfg = layout_params.to_config()
        h = ctypes.c_void_p()
        _native.check(self._lib.ocb_policy_create(ctypes.byref(self._cfg), gpu_id, hidden, n_policies, ctypes.byref(h)))
        self._h = h
        self.calls = 0

    def close(self):
        if getattr(self, "_h", None):
            self._lib.ocb_policy_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_weights(self, index: int, actor: PolicyNet = None, critic: PolicyNet = None):
        for net_id, net in ((0, actor), (1, critic)):
            if net is None:
                continue
            ts = [t.detach().to("cpu", torch.float32).contiguous() for t in
                  (net.conv_w, net.conv_b, net.fc1_w, net.fc1_b, net.fc2_w, net.fc2_b, net.head_w, net.head_b)]
            ptrs = [self._ct.c_void_p(t.data_ptr()) for t in ts]
            self._native.check(self._lib.ocb_policy_set_weights(self._h, index, net_id, *ptrs))

    def _weight_srcs(self, sets):
        """``ocb_weight_src`` array of ``set_weights_device``; checks every tensor against this handle's shapes"""
        h, co = self.hidden, self.hidden // 2
        npos = (self.layout.width - 2) * (self.layout.height - 2)
        descs = []
        for index, actor, critic in sets:
            if not 0 <= int(index) < self.n_policies:
                raise ValueError("weight set %d out of range (the handle holds %d)" % (int(index), self.n_policies))
            for net_id, net in ((0, actor), (1, critic)):
                if net is None:
                    continue
                out = NUM_ACTIONS if net_id == 0 else 1
                shapes = ((co, self.layout.channels, 3, 3), (co,), (h, co * npos), (h,), (h, h), (h,), (out, h), (out,))
                ts = [getattr(net, name) for name in _WEIGHTS]
                for name, t, shape in zip(_WEIGHTS, ts, shapes):
                    if tuple(t.shape) != shape:
                        raise ValueError("%s of set %d net %d: shape %s, expected %s" % (name, index, net_id, tuple(t.shape), shape))
                    if t.dtype != torch.float32:
                        raise ValueError("%s of set %d net %d: dtype %s, expected torch.float32" % (name, index, net_id, t.dtype))
                    if not t.is_contiguous():
                        raise ValueError("%s of set %d net %d is not contiguous" % (name, index, net_id))
                    if t.device != self.device:
                        raise ValueError("%s of set %d net %d lives on %s, the handle on %s" % (name, index, net_id, t.device,
                                                                                           self.device))
                descs.append((int(index), net_id, ts))
        if not descs:
            raise ValueError("no network to refresh")
        arr = (self._native.ocb_weight_src * len(descs))()
        for d, (index, net_id, ts) in zip(arr, descs):
            d.policy, d.net = index, net_id
            for name, t in zip(_WEIGHTS, ts):
                setattr(d, name, t.data_ptr())
        return arr

    def set_weights_device(self, sets):
        """``set_weights`` for weights already on this handle's device: ``sets`` is a sequence of ``(index, actor, critic)``
        (either net may be ``None``), packed into the same bytes ``set_weights`` writes, in ONE native call on torch's
        current stream (``ocb_policy_set_weights_device``).  Nothing synchronises, so the refresh is ordered with the
        collections around it and can be captured into a CUDA graph; the weights are read when it runs."""
        arr = self._weight_srcs(sets)
        with torch.cuda.device(self.device):
            self._native.check(self._lib.ocb_policy_set_weights_device(self._h, len(arr), arr, self._stream()))

    def read_blob(self, index: int, net: int) -> torch.Tensor:
        """the packed bytes of (weight set, net) as a uint8 device tensor (``ocb_policy_read_blob``, diagnostic)"""
        n = self._native.check(self._lib.ocb_policy_read_blob(self._h, index, net, None, 0, None))
        out = torch.empty((n,), dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self.device):
            self._native.check(self._lib.ocb_policy_read_blob(self._h, index, net, self._p(out), n, self._stream()))
        return out

    def _p(self, t):
        return None if t is None else self._ct.c_void_p(t.data_ptr())

    def _stream(self):
        return self._ct.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _rows(self, obs):
        assert obs.dtype == torch.int8 and obs.is_cuda and obs.is_contiguous()
        return obs.numel() // (self.layout.size * self.layout.channels)

    def act(self, obs, tile_policy=None, deterministic=False, seed=0, offset=None, want_logits=False, out=None):
        """obs int8 [..., W, H, C] on the device -> dict(actions int32 [M], logp f32 [M], logits f32 [M,6]|None)"""
        M = self._rows(obs)
        if out is None:
            out = {"actions": torch.empty((M,), dtype=torch.int32, device=self.device),
                   "logp": torch.empty((M,), dtype=torch.float32, device=self.device),
                   "logits": torch.empty((M, NUM_ACTIONS), dtype=torch.float32, device=self.device) if want_logits else None}
        if offset is None:
            offset = self.calls
        self.calls += 1
        with torch.cuda.device(self.device):
            self._native.check(self._lib.ocb_policy_act(self._h, self._p(obs), M, self._p(tile_policy), self._p(out["actions"]),
                                                        self._p(out["logp"]), self._p(out.get("logits")), int(deterministic),
                                                        seed, offset, self._stream()))
        return out

    def forward(self, obs, tile_policy=None, deterministic=False, seed=0, offset=None, d_offset=None,
                want_logits=False, out=None):
        """Actor and critic in ONE launch (ocb_policy_forward): dict(actions, logp, logits|None, values).
        `d_offset` is an optional device address (int) of a uint64 added to `offset` on the device."""
        M = self._rows(obs)
        if out is None:
            out = {"actions": torch.empty((M,), dtype=torch.int32, device=self.device),
                   "logp": torch.empty((M,), dtype=torch.float32, device=self.device),
                   "logits": torch.empty((M, NUM_ACTIONS), dtype=torch.float32, device=self.device) if want_logits else None,
                   "values": torch.empty((M,), dtype=torch.float32, device=self.device)}
        if offset is None:
            offset = self.calls
        self.calls += 1
        with torch.cuda.device(self.device):
            self._native.check(self._lib.ocb_policy_forward(
                self._h, self._p(obs), M, self._p(tile_policy), self._p(out["actions"]), self._p(out["logp"]),
                self._p(out.get("logits")), self._p(out["values"]), int(deterministic), seed, offset,
                self._ct.c_void_p(d_offset) if d_offset else None, self._stream()))
        return out

    def set_sampling_rows(self, rows_per_seat: int = 0, add_seat0: int = 0, add_seat1: int = 0):
        """shard-invariant sampling streams (``ocb_policy_set_sampling_rows``): for a shard of N worlds starting at
        global world ``world0`` out of ``N_total`` pass ``(N, world0, N_total - N + world0)``; ``()`` = default"""
        self._native.check(self._lib.ocb_policy_set_sampling_rows(self._h, rows_per_seat, add_seat0, add_seat1))

    def info(self) -> dict:
        r, c, b = self._ct.c_int(), self._ct.c_int(), self._ct.c_int()
        self._native.check(self._lib.ocb_policy_info(self._h, self._ct.byref(r), self._ct.byref(c), self._ct.byref(b)))
        return {"ring_slots": r.value, "chunks_per_unit": c.value, "weights_resident": r.value >= c.value,
                "smem_bytes": b.value}

    def value(self, obs, tile_policy=None, out=None):
        M = self._rows(obs)
        if out is None:
            out = torch.empty((M,), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            self._native.check(self._lib.ocb_policy_value(self._h, self._p(obs), M, self._p(tile_policy), self._p(out),
                                                          self._stream()))
        return out

    def evaluate(self, obs, actions_src, rows=None, tile_policy=None, with_critic=True, want_logits=False, out=None):
        """evaluate_actions (R_Actor.evaluate_actions r_actor_critic.py:73-109 + R_Critic.forward) over rows picked
        out of ``obs`` in place (``ocb_policy_evaluate``): obs int8 ``[..., W, H, C]`` (e.g. the whole rollout
        buffer), ``actions_src`` int32 indexed like obs rows, ``rows`` int32 ``[B]`` source-row indices (None =
        every row in order) -> dict(logp [B], entropy [B], values [B]|None, logits [B,6]|None)."""
        R = self._rows(obs)
        if rows is not None:
            assert rows.dtype == torch.int32 and rows.is_cuda and rows.is_contiguous()
        B = R if rows is None else rows.numel()
        assert actions_src.dtype == torch.int32 and actions_src.is_cuda and actions_src.is_contiguous()
        if out is None:
            f = lambda *s: torch.empty(s, dtype=torch.float32, device=self.device)
            out = {"logp": f(B), "entropy": f(B), "values": f(B) if with_critic else None,
                   "logits": f(B, NUM_ACTIONS) if want_logits else None}
        with torch.cuda.device(self.device):
            self._native.check(self._lib.ocb_policy_evaluate(
                self._h, self._p(obs), self._p(rows), B, self._p(tile_policy), self._p(actions_src), self._p(out["logp"]),
                self._p(out["entropy"]), self._p(out.get("logits")), self._p(out.get("values")), self._stream()))
        return out
