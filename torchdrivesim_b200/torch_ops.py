"""`torch.ops.tds_b200.*`: the pure-tensor entry points of libtds_b200.so registered as PyTorch custom operators
(torch.library), with their hand-written backward kernels wired in through `register_autograd` and shape functions
for fake tensors - so that they are first-class ops for `torch.compile` / `torch.export` graphs, not only Python
`autograd.Function`s.  The ops that take a static map (offroad, raster) stay in `ops.py`: a map is a library handle,
not a tensor.

    torch.ops.tds_b200.kinematic_step(state, action, lr, model, uniform_model, dt, left_handed) -> state'
    torch.ops.tds_b200.collision_pairwise(box1, box2, metric) -> overlap          (metric 0 = discs, 1 = IoU)
    torch.ops.tds_b200.collision_allpairs(ego_box, all_box, mask, metric, ego_is_prefix) -> (loss, argmax)
    torch.ops.tds_b200.agent_boxes(state, size) -> boxes
    torch.ops.tds_b200.agents_relative(absolute, n_agents, exclude_self) -> relative   (absolute [B,N,6] or [B,A,N,6])
    torch.ops.tds_b200.nearest_agents_relative(absolute, k, n_agents, max_distance) -> (relative [B,A,k,6], idx [B,A,k])
    torch.ops.tds_b200.time_to_collision(state, size, present, horizon, n_agents) -> (ttc [B,A], idx [B,A])

This module holds the registrations only: every operator body calls the launcher of ops.py that the autograd Functions
use too, so both check their inputs and launch the kernels the same way.

Reference call sites: kinematic.py:462-523, infractions.py:503-545 / 307-324, simulator.py:1161-1194, 748-821.
"""
from typing import Optional, Tuple

import torch
from torch import Tensor

from . import ops

_NS = "tds_b200"


# ------------------------------------------------------------------------------------ kinematic step
@torch.library.custom_op(f"{_NS}::kinematic_step", mutates_args=())
def kinematic_step(state: Tensor, action: Tensor, lr: Tensor, model: Optional[Tensor], uniform_model: int, dt: float,
                   left_handed: bool) -> Tensor:
    return ops._kinematic_fwd(state, action, lr, model, uniform_model, ops.kinematic_params(dt=dt, left_handed=left_handed))


@kinematic_step.register_fake
def _(state, action, lr, model, uniform_model, dt, left_handed):
    return torch.empty_like(state, dtype=torch.float32)


@torch.library.custom_op(f"{_NS}::kinematic_step_backward", mutates_args=())
def kinematic_step_backward(grad_out: Tensor, state: Tensor, action: Tensor, lr: Tensor, model: Optional[Tensor], uniform_model: int,
                            dt: float, left_handed: bool) -> Tuple[Tensor, Tensor, Tensor]:
    return ops._kinematic_bwd(state, action, lr, model, uniform_model, ops.kinematic_params(dt=dt, left_handed=left_handed),
                              grad_out)


@kinematic_step_backward.register_fake
def _(grad_out, state, action, lr, model, uniform_model, dt, left_handed):
    return (torch.empty_like(state, dtype=torch.float32), torch.empty_like(action, dtype=torch.float32),
            torch.empty_like(lr, dtype=torch.float32))


def _kin_setup(ctx, inputs, output):
    state, action, lr, model, uniform_model, dt, left_handed = inputs
    ctx.save_for_backward(state, action, lr, model)
    ctx.meta = (uniform_model, dt, left_handed)


def _kin_backward(ctx, grad_out):
    state, action, lr, model = ctx.saved_tensors
    gs, ga, gl = kinematic_step_backward(grad_out.contiguous(), state, action, lr, model, *ctx.meta)
    return gs, ga, gl, None, None, None, None


kinematic_step.register_autograd(_kin_backward, setup_context=_kin_setup)


# ------------------------------------------------------------------------------------ collisions
@torch.library.custom_op(f"{_NS}::collision_pairwise", mutates_args=())
def collision_pairwise(box1: Tensor, box2: Tensor, metric: int) -> Tensor:
    return ops._pairwise_fwd(box1, box2, metric)


@collision_pairwise.register_fake
def _(box1, box2, metric):
    return box1.new_empty(box1.shape[:-1], dtype=torch.float32)


@torch.library.custom_op(f"{_NS}::collision_pairwise_backward", mutates_args=())
def collision_pairwise_backward(grad_out: Tensor, box1: Tensor, box2: Tensor, metric: int) -> Tuple[Tensor, Tensor]:
    return ops._pairwise_bwd(box1, box2, metric, grad_out)


@collision_pairwise_backward.register_fake
def _(grad_out, box1, box2, metric):
    return torch.empty_like(box1, dtype=torch.float32), torch.empty_like(box2, dtype=torch.float32)


collision_pairwise.register_autograd(
    lambda ctx, g: (*collision_pairwise_backward(g.contiguous(), *ctx.saved_tensors, ctx.metric), None),
    setup_context=lambda ctx, inputs, output: (ctx.save_for_backward(inputs[0], inputs[1]), setattr(ctx, "metric", inputs[2])))


@torch.library.custom_op(f"{_NS}::collision_allpairs", mutates_args=())
def collision_allpairs(ego_box: Tensor, all_box: Tensor, mask: Tensor, metric: int, ego_is_prefix: bool) -> Tuple[Tensor, Tensor]:
    return ops._allpairs_fwd(ego_box, all_box, mask, metric, ego_is_prefix)


@collision_allpairs.register_fake
def _(ego_box, all_box, mask, metric, ego_is_prefix):
    shape = ego_box.shape[:2]
    return ego_box.new_empty(shape, dtype=torch.float32), ego_box.new_empty(shape, dtype=torch.int32)


@torch.library.custom_op(f"{_NS}::collision_allpairs_backward", mutates_args=())
def collision_allpairs_backward(grad_out: Tensor, ego_box: Tensor, all_box: Tensor, mask: Tensor, argmax: Tensor, metric: int,
                                ego_is_prefix: bool) -> Tuple[Tensor, Tensor]:
    return ops._allpairs_bwd(ego_box, all_box, mask, metric, ego_is_prefix, argmax, grad_out)


@collision_allpairs_backward.register_fake
def _(grad_out, ego_box, all_box, mask, argmax, metric, ego_is_prefix):
    return torch.empty_like(ego_box, dtype=torch.float32), torch.empty_like(all_box, dtype=torch.float32)


def _ap_setup(ctx, inputs, output):
    ego, allb, mask, metric, prefix = inputs
    ctx.save_for_backward(ego, allb, mask, output[1])
    ctx.meta = (metric, prefix)
    ctx.mark_non_differentiable(output[1])


def _ap_backward(ctx, g_out, g_arg):
    ego, allb, mask, arg = ctx.saved_tensors
    ge, ga = collision_allpairs_backward(g_out.contiguous(), ego, allb, mask, arg, *ctx.meta)
    return ge, ga, None, None, None


collision_allpairs.register_autograd(_ap_backward, setup_context=_ap_setup)


# ------------------------------------------------------------------------------------ boxes
@torch.library.custom_op(f"{_NS}::agent_boxes", mutates_args=())
def agent_boxes(state: Tensor, size: Tensor) -> Tensor:
    return ops._agent_boxes(state, size)


@agent_boxes.register_fake
def _(state, size):
    return state.new_empty(state.shape[:-1] + (5,), dtype=torch.float32)


agent_boxes.register_autograd(lambda ctx, g: ops._agent_boxes_grad(g, ctx.size_cols),
                              setup_context=lambda ctx, inputs, output: setattr(ctx, "size_cols", inputs[1].shape[-1]))


# ------------------------------------------------------------------------------------ relative observations
@torch.library.custom_op(f"{_NS}::agents_relative", mutates_args=())
def agents_relative(absolute: Tensor, n_agents: Optional[int], exclude_self: bool) -> Tensor:
    return ops._agents_relative_fwd(absolute, n_agents, exclude_self)


@agents_relative.register_fake
def _(absolute, n_agents, exclude_self):
    B, A, N, M = ops._agents_relative_shape(absolute, n_agents, exclude_self)
    return absolute.new_empty((B, A, M, 6), dtype=torch.float32)


@torch.library.custom_op(f"{_NS}::agents_relative_backward", mutates_args=())
def agents_relative_backward(grad_out: Tensor, absolute: Tensor, n_agents: Optional[int], exclude_self: bool) -> Tensor:
    return ops._agents_relative_bwd(absolute, n_agents, exclude_self, grad_out)


@agents_relative_backward.register_fake
def _(grad_out, absolute, n_agents, exclude_self):
    return torch.empty_like(absolute, dtype=torch.float32)


agents_relative.register_autograd(
    lambda ctx, g: (agents_relative_backward(g.contiguous(), *ctx.saved_tensors, *ctx.meta), None, None),
    setup_context=lambda ctx, inputs, output: (ctx.save_for_backward(inputs[0]), setattr(ctx, "meta", inputs[1:])))


@torch.library.custom_op(f"{_NS}::nearest_agents_relative", mutates_args=())
def nearest_agents_relative(absolute: Tensor, k: int, n_agents: Optional[int], max_distance: float) -> Tuple[Tensor, Tensor]:
    return ops._nearest_fwd(absolute, k, n_agents, max_distance)


@nearest_agents_relative.register_fake
def _(absolute, k, n_agents, max_distance):
    B, A, N, k = ops._nearest_shape(absolute, k, n_agents)
    ops._nearest_r2(max_distance)
    return absolute.new_empty((B, A, k, 6), dtype=torch.float32), absolute.new_empty((B, A, k), dtype=torch.int64)


@torch.library.custom_op(f"{_NS}::nearest_agents_relative_backward", mutates_args=())
def nearest_agents_relative_backward(grad_out: Tensor, absolute: Tensor, idx: Tensor, k: int, n_agents: Optional[int]) -> Tensor:
    return ops._nearest_bwd(absolute, k, n_agents, idx, grad_out)


@nearest_agents_relative_backward.register_fake
def _(grad_out, absolute, idx, k, n_agents):
    return torch.empty_like(absolute, dtype=torch.float32)


def _nearest_setup(ctx, inputs, output):
    absolute, k, n_agents, max_distance = inputs
    ctx.save_for_backward(absolute, output[1])
    ctx.meta = (k, n_agents)
    ctx.mark_non_differentiable(output[1])


def _nearest_backward(ctx, g_out, g_idx):
    absolute, idx = ctx.saved_tensors
    return nearest_agents_relative_backward(g_out.contiguous(), absolute, idx, *ctx.meta), None, None, None


nearest_agents_relative.register_autograd(_nearest_backward, setup_context=_nearest_setup)


# ------------------------------------------------------------------------------------ time to collision
@torch.library.custom_op(f"{_NS}::time_to_collision", mutates_args=())
def time_to_collision(state: Tensor, size: Tensor, present: Tensor, horizon: float, n_agents: Optional[int]) -> Tuple[Tensor, Tensor]:
    return ops._time_to_collision_fwd(state, size, present, n_agents, horizon)


@time_to_collision.register_fake
def _(state, size, present, horizon, n_agents):
    B, A, N, H = ops._ttc_shape(state, size, present, n_agents, horizon)
    return state.new_empty((B, A), dtype=torch.float32), state.new_empty((B, A), dtype=torch.int64)


@torch.library.custom_op(f"{_NS}::time_to_collision_backward", mutates_args=())
def time_to_collision_backward(grad_out: Tensor, state: Tensor, size: Tensor, present: Tensor, idx: Tensor, horizon: float,
                               n_agents: Optional[int]) -> Tuple[Tensor, Tensor]:
    return ops._time_to_collision_bwd(state, size, present, n_agents, horizon, idx, grad_out)


@time_to_collision_backward.register_fake
def _(grad_out, state, size, present, idx, horizon, n_agents):
    return torch.empty_like(state, dtype=torch.float32), torch.empty_like(size, dtype=torch.float32)


def _ttc_setup(ctx, inputs, output):
    state, size, present, horizon, n_agents = inputs
    ctx.save_for_backward(state, size, present, output[1])
    ctx.meta = (horizon, n_agents)
    ctx.mark_non_differentiable(output[1])


def _ttc_backward(ctx, g_ttc, g_idx):
    state, size, present, idx = ctx.saved_tensors
    gs, gz = time_to_collision_backward(g_ttc.contiguous(), state, size, present, idx, *ctx.meta)
    return gs, gz, None, None, None


time_to_collision.register_autograd(_ttc_backward, setup_context=_ttc_setup)
