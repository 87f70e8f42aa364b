"""Controller observation + actor forward on the device (SURVEY.md 8(f)-2).

Mirrors ``ControlInterface.get_observation`` (models/controller/rl_pose.py:173-187) and
``ActorCritic.act_inference`` (algo/ppo/ppo/module.py:89-91) of the reference: with the view ring
(:mod:`rgbmanip_b200.view_ring`) the pose / mask-box history already lives on the GPU, so the ``[N, 60]`` observation and
the 60 -> 96 -> 96 -> 32 -> 12 ELU policy run as one small kernel on the estimator's stream instead of a host round trip.
The predicted box is not an actor input (rl_pose.py:177-178 is commented out in the reference)."""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib as L


ACTIVATIONS = {"elu": 0, "selu": 1, "relu": 2, "crelu": 2, "lrelu": 3, "tanh": 4, "sigmoid": 5}   # module.py:110-126


class DeviceActor:
    def __init__(self, actor_state_dict, ring, activation="elu"):
        """actor_state_dict: the ``actor.*`` entries of the reference's ActorCritic state dict (nn.Sequential of
        Linear/activation); ``activation``: ``model_cfg['activation']`` of the policy (cfg/controller/rl.yaml: elu)."""
        if activation not in ACTIVATIONS:
            raise ValueError(f"unsupported actor activation {activation!r} (the reference's get_activation knows {sorted(ACTIVATIONS)})")
        self.activation = ACTIVATIONS[activation]
        self.lib = L.load()
        self.ring = ring
        self.shards = None
        if hasattr(ring, "shards"):
            # a ring sharded over devices: the weights are replicated on every shard's device and each shard's actor reads its
            # own queues (an observation depends on its environment's queues and the step only)
            self.shards = [DeviceActor(actor_state_dict, s, activation) for s in ring.shards]
            self.dims = self.shards[0].dims
            return
        dev = ring.device
        sd = {k.replace("actor_critic.", ""): v for k, v in actor_state_dict.items()}
        idx = sorted({int(k.split(".")[1]) for k in sd if k.startswith("actor.") and k.endswith(".weight")})
        if not idx:
            raise KeyError("no actor.* Linear layers in the state dict")
        t = lambda a: torch.as_tensor(np.asarray(a.detach().cpu() if hasattr(a, "detach") else a)).float().to(dev).contiguous()
        self.W = [t(sd[f"actor.{i}.weight"]) for i in idx]
        self.b = [t(sd[f"actor.{i}.bias"]) for i in idx]
        self.dims = [self.W[0].shape[1]] + [w.shape[0] for w in self.W]
        if self.dims[0] != ring.max_steps * 12:
            raise ValueError(f"actor expects {self.dims[0]} inputs, the ring provides {ring.max_steps * 12}")
        n = len(self.W)
        self._dims = (C.c_int32 * (n + 1))(*self.dims)
        self._wp = (C.c_void_p * n)(*[w.data_ptr() for w in self.W])
        self._bp = (C.c_void_p * n)(*[b.data_ptr() for b in self.b])
        self.obs = torch.zeros((ring.num_envs, self.dims[0]), dtype=torch.float32, device=dev)
        self.act = torch.zeros((ring.num_envs, self.dims[-1]), dtype=torch.float32, device=dev)

    def act_inference(self, accumulate_steps=None):
        """-> (actions [N, A], observation [N, T*12]) device tensors for the ring's current queues."""
        r = self.ring
        step = (r.accumulate_steps if accumulate_steps is None else accumulate_steps) - 1
        if not 0 <= step < r.max_steps:
            raise IndexError(f"one_hot index {step} outside [0, {r.max_steps})")       # torch.nn.functional.one_hot raises too
        if self.shards is not None:          # -> [N, A] / [N, T*12] in env order on the first device
            outs = []
            for a in self.shards:
                with torch.cuda.device(a.ring.device):
                    outs.append(a.act_inference(step + 1))
            return tuple(torch.cat([o[i].to(r.device) for o in outs]) for i in (0, 1))
        st = C.c_void_p(torch.cuda.current_stream(r.device).cuda_stream)
        L.check(self.lib.adp_actor_forward(L.ptr(r.pose), L.ptr(r.bbox), r.max_steps, r.num_envs, step, len(self.W), self._dims,
                                           self._wp, self._bp, self.activation, L.ptr(self.obs), L.ptr(self.act), st), "actor_forward")
        return self.act, self.obs

    def get_observation(self):
        return self.act_inference()[1]
