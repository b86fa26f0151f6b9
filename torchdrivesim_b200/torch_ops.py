"""`torch.ops.tds_b200.*`: the pure-tensor entry points of libtds_b200.so registered as PyTorch custom operators
(torch.library), with their hand-written backward kernels wired in through `register_autograd` and shape functions
for fake tensors - so that they are first-class ops for `torch.compile` / `torch.export` graphs, not only Python
`autograd.Function`s.  The ops that take a static map (offroad, raster) stay in `ops.py`: a map is a library handle,
not a tensor.

    torch.ops.tds_b200.kinematic_step(state, action, lr, model, uniform_model, dt, left_handed) -> state'
    torch.ops.tds_b200.collision_pairwise(box1, box2, metric) -> overlap          (metric 0 = discs, 1 = IoU)
    torch.ops.tds_b200.collision_allpairs(ego_box, all_box, mask, metric, ego_is_prefix) -> (loss, argmax)
    torch.ops.tds_b200.agent_boxes(state, size) -> boxes

This module holds the registrations only: every operator body calls the launcher of ops.py that the autograd Functions
use too, so both check their inputs and launch the kernels the same way.

Reference call sites: kinematic.py:462-523, infractions.py:503-545 / 307-324, simulator.py:1161-1194.
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
