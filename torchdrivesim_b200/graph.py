"""CUDA-graph replay of the whole hot path.

`GraphedHotPath` records ONE step of a `Simulator` (kinematic step -> egocentric birdviews -> collisions ->
offroad) into a CUDA graph over static buffers and replays it with new actions; collisions and offroad are a second
branch of the graph that runs beside the birdviews.  The step consists of ~5 of
our kernels plus a dozen tiny torch kernels; replaying a graph removes the eager-mode launch gaps between
them (the reference has no equivalent: it is eager PyTorch + a Python loop per triangle).

Inference-only (no autograd tape is recorded); differentiable rollouts have their own graph (`FusedRollout`).

A graph reads and writes FIXED buffers.  Everything the step reads is therefore moved into buffers this class owns
(traffic-control states, NPC states, waypoint-goal masks and states) and refreshed in place; tensors the caller swaps
into the simulator afterwards (`update_present_mask`, a new `waypoint_goals.mask`) are invisible to the graph - update
`sim.present_mask` / the goal buffers in place (`.copy_`) instead.
"""
from typing import Optional, Tuple

import torch
from torch import Tensor

from . import _lib
from .rendering import Resolution
from .simulator import Simulator


class GraphedHotPath:
    def __init__(self, sim: Simulator, res: Optional[Resolution] = None, fov: Optional[float] = None,
                 render: bool = True, warmup: int = 2):
        self.sim = sim
        state = sim.get_state()
        if not state.is_cuda:
            raise _lib.TdsError("GraphedHotPath needs a Simulator on a CUDA device")
        dev = state.device
        B, A = state.shape[0], state.shape[1]
        res = sim.renderer.res if res is None else res
        self.action = torch.zeros(B, A, sim.action_size, dtype=torch.float32, device=dev)
        self.state = state.detach().clone()
        self.images = torch.empty(B, A, 3, res.height, res.width, dtype=torch.float32, device=dev) if render else None
        self.collision = torch.empty(B, A, dtype=torch.float32, device=dev)
        self.offroad = torch.empty(B, A, dtype=torch.float32, device=dev)
        self._res, self._fov, self._render = res, fov, render
        # traffic-control states change between steps: the graph reads them from static buffers
        self._control_state = {}
        for name, control in (sim.traffic_controls or {}).items():
            buf = control.state.detach().clone()
            control.set_state(buf)
            self._control_state[name] = buf
        # so do the NPCs: the controller advances eagerly (one launch) into static buffers
        self._npc_state = self._npc_present = None
        if sim.npc_count > 0:
            self._npc_state = sim.npc_controller.npc_state.detach().to(torch.float32).clone()
            self._npc_present = sim.npc_controller.npc_present_mask.detach().clone()
            sim.npc_controller.npc_state, sim.npc_controller.npc_present_mask = self._npc_state, self._npc_present
        # ... and the waypoint goals: their step (simulator.py:860-861) is part of the graph and updates these in place
        self._goals = sim.waypoint_goals
        if self._goals is not None:
            self._goals.mask = self._goals.mask.to(torch.bool).contiguous().clone()
            self._goals.state = self._goals.state.to(torch.int64).contiguous().clone()
            self._goal_saved = (self._goals.mask.clone(), self._goals.state.clone())
        sim.kinematic_model.set_state(self.state)
        self._side = torch.cuda.Stream(device=dev)
        # warm up on a side stream (allocator, lazily built map handles), then capture
        s = torch.cuda.Stream(device=dev)
        s.wait_stream(torch.cuda.current_stream(dev))
        saved = self.state.clone()
        with torch.cuda.stream(s), torch.no_grad():
            for _ in range(max(warmup, 1)):
                self._body()
        torch.cuda.current_stream(dev).wait_stream(s)
        torch.cuda.synchronize(dev)
        self._restore(saved)
        self.graph = torch.cuda.CUDAGraph()
        # captured on the stream of the warm-up: the library keys its scratch buffers by (device, stream), and a buffer
        # that the warm-up allocated must be the one the captured kernels find
        with torch.no_grad(), torch.cuda.graph(self.graph, stream=s):
            self._body()
        self._restore(saved)

    def _restore(self, saved: Tensor) -> None:
        self.state.copy_(saved)
        if self._goals is not None:
            self._goals.mask.copy_(self._goal_saved[0])
            self._goals.state.copy_(self._goal_saved[1])

    def _body(self) -> None:
        sim = self.sim
        sim.kinematic_model.set_state(self.state)
        # Simulator.step minus the host-side control / NPC stepping; the state is updated in place: the graph chains
        # steps through this static buffer
        sim.kinematic_model.step(self.action, out=self.state)
        if self._goals is not None:
            self._goals.step(self.state, sim.internal_time, threshold=sim.cfg.waypoint_removal_threshold, in_place=True)
        if not self._render:
            sim.compute_collision(out=self.collision)
            sim.compute_offroad(out=self.offroad)
            return
        # collisions and offroad depend on the new state only: a second branch of the graph, beside the raster.  Neither
        # touches the raster's scratch buffers, which the library keys by (device, stream) and finds on the main stream.
        main = torch.cuda.current_stream()
        self._side.wait_stream(main)
        with torch.cuda.stream(self._side):
            sim.compute_collision(out=self.collision)
            sim.compute_offroad(out=self.offroad)
        sim.render_egocentric(res=self._res, fov=self._fov, out=self.images)
        main.wait_stream(self._side)

    def run(self, action: Tensor) -> Tuple[Optional[Tensor], Tensor, Tensor]:
        """One step with `action` [B,A,Ac] (device or pinned host tensor).  Returns the static output
        buffers (images, collision, offroad); they are overwritten by the next call."""
        self.action.copy_(action, non_blocking=True)
        self.sim.internal_time += 1
        for name, control in (self.sim.traffic_controls or {}).items():
            control.step(self.sim.internal_time)     # host-side rule (replay tensor or compute_state) ...
            buf = self._control_state[name]
            if control.state is not buf:
                buf.copy_(control.state)             # ... lands in the buffer the graph reads
                control.set_state(buf)
        if self._npc_state is not None:
            ctrl = self.sim.npc_controller
            ctrl.advance_npcs(self.sim)
            if ctrl.npc_state is not self._npc_state:
                self._npc_state.copy_(ctrl.npc_state)
                self._npc_present.copy_(ctrl.npc_present_mask)
                ctrl.npc_state, ctrl.npc_present_mask = self._npc_state, self._npc_present
        self.graph.replay()
        return self.images, self.collision, self.offroad

    def set_state(self, state: Tensor) -> None:
        self.state.copy_(state)
