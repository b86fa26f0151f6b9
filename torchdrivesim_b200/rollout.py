"""Differentiable rollouts as ONE CUDA graph (BASELINE config 5: "20-step rollout with backward through kinematics +
collision loss", examples/imitation_learning.py:279-335 in the reference).

Through autograd a T-step rollout is ~30 small launches per step: every `Simulator.step` / `compute_collision` /
`compute_offroad` is a custom autograd Function around a 5 us kernel, plus torch glue (cat, sum, pow, mean) and their
backward nodes - the GPU idles between launches.  `FusedRollout` issues the same kernels through the same launchers of
ops.py in a fixed order, forward and backward, into static buffers and records the sequence once.  Its inputs are kept
in the kernels' dtypes (the present mask as bool), so the launchers pass them through without a copy; only the loss
and the gradient merge call the C ABI directly:

    forward,  t = 0..T-1:  kinematic step -> boxes -> all-pairs collision -> offroad -> loss accumulation
    backward, t = T-1..0:  offroad backward, collision backward -> merge with the gradient from step t+1 and the
                           target term (tds_rollout_grad) -> kinematic backward (-> d loss / d action[t])

    loss = sum_t [ w_collision * sum(collision_t) + w_offroad * sum(offroad_t) + w_target * mean((xy_t - target)^2) ]

The gradients are those the eager path (`ops.*` autograd Functions) produces; tests/test_gpu_rollout.py checks them
against it and against the oracle's torch-autograd restatement.
"""
from typing import Optional, Tuple

import torch
from torch import Tensor

from . import _lib, ops
from .maps import MapSet, StaticMap


class FusedRollout:
    def __init__(self, road, state0: Tensor, agent_size: Tensor, lr: Tensor, present_mask: Tensor, steps: int,
                 offroad_threshold: float = 0.5, left_handed: bool = False, target_xy: Optional[Tensor] = None,
                 w_collision: float = 1.0, w_offroad: float = 1.0, w_target: float = 1.0,
                 collision_metric: int = _lib.METRIC_DISCS, model: Optional[Tensor] = None,
                 uniform_model: int = _lib.MODEL_BICYCLE, dt: float = 0.1, warmup: int = 2):
        if not state0.is_cuda:
            raise _lib.TdsError("FusedRollout needs CUDA tensors: there is no CPU implementation")
        self.lib = _lib.load()
        self.mapset = road if isinstance(road, MapSet) else MapSet([road])
        dev = state0.device
        self.dev = dev
        B, A = state0.shape[0], state0.shape[1]
        self.B, self.A, self.T = B, A, int(steps)
        n = B * A
        f32 = dict(dtype=torch.float32, device=dev)
        self.state = torch.empty(self.T + 1, B, A, 4, **f32)          # the whole trajectory is kept for the backward
        self.state[0].copy_(_lib.as_f32(state0))
        self.size = _lib.as_f32(agent_size[..., :2]).clone()
        self.lr = _lib.as_f32(lr).clone()
        self.present = (present_mask.detach() != 0).contiguous()     # bool: the launchers view it as uint8, no copy
        self.model = None if model is None else _lib.as_i32(model).clone()
        self.uniform_model = int(uniform_model)
        self.params = ops.kinematic_params(dt=dt, left_handed=left_handed)
        self.metric = int(collision_metric)
        self.threshold = float(offroad_threshold)
        self.target = None if target_xy is None else _lib.as_f32(target_xy).clone()
        self.w = (float(w_collision), float(w_offroad), float(w_target))
        self.actions = torch.zeros(self.T, B, A, 2, **f32)
        self.box = torch.empty(self.T, B, A, 5, **f32)
        self.argmax = torch.empty(self.T, B, A, dtype=torch.int32, device=dev)
        self.face = torch.empty(self.T, B, A, 4, dtype=torch.int32, device=dev)
        self.collision = torch.empty(B, A, **f32)
        self.offroad = torch.empty(B, A, **f32)
        self.acc = torch.zeros(3, dtype=torch.float64, device=dev)
        self.ones = torch.ones(B, A, **f32)
        self.g_off = torch.empty(B, A, 4, **f32)
        self.g_ego = torch.empty(B, A, 5, **f32)
        self.g_all = torch.empty(B, A, 5, **f32)
        self.g_state = [torch.empty(B, A, 4, **f32) for _ in range(2)]
        self.g_merged = torch.empty(B, A, 4, **f32)
        self.grad_actions = torch.empty(self.T, B, A, 2, **f32)
        self.loss = torch.zeros((), **f32)
        n_agents = B * A
        self._scale = torch.tensor([self.w[0], self.w[1], 0.0 if self.target is None else self.w[2] / (2 * n_agents)],
                                   dtype=torch.float64, device=dev)
        # warm up on a side stream (lazily built map handles, allocator), then capture
        s = torch.cuda.Stream(device=dev)
        s.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(s), torch.no_grad():
            for _ in range(max(warmup, 1)):
                self._body()
        torch.cuda.current_stream(dev).wait_stream(s)
        torch.cuda.synchronize(dev)
        self.graph = torch.cuda.CUDAGraph()
        # captured on the stream of the warm-up: the library keys its scratch buffers by (device, stream), and a buffer
        # that the warm-up allocated must be the one the captured kernels find
        with torch.no_grad(), torch.cuda.graph(self.graph, stream=s):
            self._body()

    # ---- the fixed launch sequence (eager during warm-up, recorded once) --------------------------------------
    def _body(self) -> None:
        lib, p, st = self.lib, _lib.ptr, _lib.stream_ptr(self.dev)
        B, A, T = self.B, self.A, self.T
        n = B * A
        wc, wo, wt = self.w
        # the target term is w_t * mean over (agents, xy) of the squared error = w_t / (2 n) * sum |xy - target|^2
        wt_grad = 0.0 if self.target is None else wt / n
        kin = (self.lr, self.model, self.uniform_model, self.params)
        off = (self.size, self.present, self.mapset, self.threshold)
        self.acc.zero_()
        for t in range(T):
            s0, s1 = self.state[t], self.state[t + 1]
            ops._kinematic_fwd(s0, self.actions[t], *kin, out=s1)
            ops._agent_boxes(s1, self.size, out=self.box[t])
            ops._allpairs_fwd(self.box[t], self.box[t], self.present, self.metric, True, out=(self.collision, self.argmax[t]))
            ops._offroad_fwd(s1, *off, out=(self.offroad, self.face[t]))
            _lib.check(lib.tds_rollout_loss(p(self.collision), p(self.offroad), p(s1), p(self.target), n, p(self.acc), st))
        self.loss.copy_((self.acc * self._scale).sum())
        g_next = None
        for t in range(T - 1, -1, -1):
            s0, s1 = self.state[t], self.state[t + 1]
            ops._offroad_bwd(s1, *off, self.face[t], self.ones, out=(self.g_off, None))
            ops._allpairs_bwd(self.box[t], self.box[t], self.present, self.metric, True, self.argmax[t], self.ones,
                              out=(self.g_ego, self.g_all))
            _lib.check(lib.tds_rollout_grad(None if g_next is None else p(g_next), p(self.g_off), p(self.g_ego), p(self.g_all),
                                            p(s1), p(self.target), wo, wc, wt_grad, n, p(self.g_merged), st))
            g_out = self.g_state[t & 1]
            ops._kinematic_bwd(s0, self.actions[t], *kin, self.g_merged, out=(g_out, self.grad_actions[t], None))
            g_next = g_out
        self.grad_state0 = g_next

    def run(self, actions: Tensor, state0: Optional[Tensor] = None) -> Tuple[Tensor, Tensor]:
        """actions [T,B,A,2] (device or pinned host) -> (loss, d loss / d actions [T,B,A,2]); both are static buffers
        that the next call overwrites.  `state0` replaces the initial state when given."""
        if tuple(actions.shape) != tuple(self.actions.shape):
            raise _lib.TdsError(f"actions must be {list(self.actions.shape)}")
        self.actions.copy_(actions.detach(), non_blocking=True)
        if state0 is not None:
            self.state[0].copy_(state0.detach(), non_blocking=True)
        self.graph.replay()
        return self.loss, self.grad_actions

    @property
    def trajectory(self) -> Tensor:
        """[T+1,B,A,4]: the states of the last rollout (static buffer)."""
        return self.state
