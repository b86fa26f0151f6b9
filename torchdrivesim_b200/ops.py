"""Functional ops over libtds_b200.so with autograd wiring (kinematics, collisions, offroad, raster, observations).

Every function takes CUDA tensors in the reference's layouts and launches on the current torch
stream.  Nothing here has a CPU implementation; `_lib.ptr` raises on CPU tensors.

The differentiable kernels (kinematic step, pairwise and all-pairs collision, agent boxes, relative and nearest-agent
observations, nearest map segments, range scan, time to collision, offroad) are launched by one private launcher per
entry point (`_kinematic_fwd` ... `_offroad_bwd`).  The autograd Functions and `out=` paths here,
the custom operators of torch_ops.py and `FusedRollout` all call them.  A launcher checks that the shapes of its inputs
agree before it touches the library, converts them with the `_lib.as_*` helpers (an input already in the kernel's dtype
and contiguous is passed through without a copy, which CUDA-graph capture relies on), allocates the outputs it is not
given and launches on the current stream.
"""
import ctypes
import math
import operator
from typing import Optional, Tuple

import torch

from . import _lib
from .maps import MapSet

_F32_HALF_PI = 1.5707963705062866  # float32(pi / 2), the reference's _normalization_factor (kinematic.py:420)


def kinematic_params(dt: float = 0.1, max_acceleration: float = 5.0, max_steering: float = math.pi / 2,
                     max_yaw_rate: float = math.pi / 2, left_handed: bool = False, max_dx: float = 20.0,
                     max_dpsi: float = 10 * math.pi, max_dv: float = 5.0) -> "_lib.KinematicParams":
    return _lib.KinematicParams(dt, max_acceleration, max_steering, max_yaw_rate, 1 if left_handed else 0,
                                max_dx, max_dpsi, max_dv)


# ------------------------------------------------------------------------------------ kinematics
def _check_out(out: torch.Tensor, shape, what: str) -> None:
    if out.dtype != torch.float32 or not out.is_contiguous() or tuple(out.shape) != tuple(shape):
        raise _lib.TdsError(f"{what}: `out` must be a contiguous float32 tensor of shape {list(shape)}")


def _kinematic_inputs(state, action, lr, model):
    adim = action.shape[-1]
    if adim not in (2, 4):
        raise _lib.TdsError("kinematic_step: the action must have 2 or 4 values per agent")
    s = _lib.as_f32(state).reshape(-1, 4)
    a = _lib.as_f32(action).reshape(-1, adim)
    l = None if lr is None else _lib.as_f32(lr).reshape(-1)
    m = None if model is None else _lib.as_i32(model).reshape(-1)
    n = s.shape[0]
    if a.shape[0] != n or (l is not None and l.shape[0] != n) or (m is not None and m.shape[0] != n):
        raise _lib.TdsError("kinematic_step: state, action, lr and model must agree on the batch shape")
    return s, a, l, m


def _kinematic_fwd(state, action, lr, model, uniform_model, params, out=None):
    """-> the new state, written into `out` when given (which may alias `state`)."""
    s, a, l, m = _kinematic_inputs(state, action, lr, model)
    if out is None:
        out = torch.empty(state.shape, dtype=torch.float32, device=s.device)
    else:
        _check_out(out, state.shape, "kinematic_step")
    _lib.check(_lib.load().tds_kinematic_step_fwd(_lib.ptr(s), _lib.ptr(a), a.shape[1], _lib.ptr(l), _lib.ptr(m), uniform_model,
                                                  s.shape[0], ctypes.byref(params), _lib.ptr(out), _lib.stream_ptr(s.device)))
    return out


def _kinematic_bwd(state, action, lr, model, uniform_model, params, grad, out=None):
    """-> (d state, d action, d lr); `out` holds the three buffers, None for a gradient that is not wanted."""
    s, a, l, m = _kinematic_inputs(state, action, lr, model)
    g = _lib.as_f32(grad)
    if out is None:
        out = (torch.empty(state.shape, dtype=torch.float32, device=s.device),
               torch.empty(action.shape, dtype=torch.float32, device=s.device),
               None if lr is None else torch.empty(lr.shape, dtype=torch.float32, device=s.device))
    gs, ga, gl = out
    _lib.check(_lib.load().tds_kinematic_step_bwd(_lib.ptr(s), _lib.ptr(a), a.shape[1], _lib.ptr(l), _lib.ptr(m), uniform_model,
                                                  s.shape[0], ctypes.byref(params), _lib.ptr(g), _lib.ptr(gs), _lib.ptr(ga),
                                                  _lib.ptr(gl), _lib.stream_ptr(s.device)))
    return out


class _KinematicStep(torch.autograd.Function):
    @staticmethod
    def forward(ctx, state, action, lr, model, uniform_model, params):
        ctx.save_for_backward(state, action, lr, model)
        ctx.meta = (uniform_model, params)
        return _kinematic_fwd(state, action, lr, model, uniform_model, params)

    @staticmethod
    def backward(ctx, grad_out):
        return (*_kinematic_bwd(*ctx.saved_tensors, *ctx.meta, grad_out), None, None, None)


def kinematic_step(state: torch.Tensor, action: torch.Tensor, lr: Optional[torch.Tensor],
                   model: Optional[torch.Tensor] = None, uniform_model: int = _lib.MODEL_BICYCLE,
                   params: Optional["_lib.KinematicParams"] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """state [...,4], action [...,2|4], lr [...], model [...] int (or None: `uniform_model`) -> new state.
    `out` (contiguous float32, the state's shape; may alias `state`): written directly, no autograd tape."""
    params = params or kinematic_params()
    if out is None:
        return _KinematicStep.apply(state, action, lr, model, uniform_model, params)
    return _kinematic_fwd(state, action, lr, model, uniform_model, params, out)


# ------------------------------------------------------------------------------------ collisions
def _pairwise_inputs(box1, box2):
    if box1.shape != box2.shape or box1.shape[-1] != 5:
        raise _lib.TdsError("collision_pairwise: boxes must have identical shape [...,5]")
    return _lib.as_f32(box1), _lib.as_f32(box2)


def _pairwise_fwd(box1, box2, metric):
    b1, b2 = _pairwise_inputs(box1, box2)
    out = torch.empty(b1.shape[:-1], dtype=torch.float32, device=b1.device)
    _lib.check(_lib.load().tds_collision_pairwise_fwd(_lib.ptr(b1), _lib.ptr(b2), out.numel(), metric, _lib.ptr(out),
                                                      _lib.stream_ptr(b1.device)))
    return out


def _pairwise_bwd(box1, box2, metric, grad):
    b1, b2 = _pairwise_inputs(box1, box2)
    g = _lib.as_f32(grad)
    g1, g2 = torch.empty_like(b1), torch.empty_like(b2)
    _lib.check(_lib.load().tds_collision_pairwise_bwd(_lib.ptr(b1), _lib.ptr(b2), b1.numel() // 5, metric, _lib.ptr(g),
                                                      _lib.ptr(g1), _lib.ptr(g2), _lib.stream_ptr(b1.device)))
    return g1, g2


class _Pairwise(torch.autograd.Function):
    @staticmethod
    def forward(ctx, box1, box2, metric):
        ctx.save_for_backward(box1, box2)
        ctx.metric = metric
        return _pairwise_fwd(box1, box2, metric)

    @staticmethod
    def backward(ctx, grad_out):
        return (*_pairwise_bwd(*ctx.saved_tensors, ctx.metric, grad_out), None)


def collision_pairwise(box1: torch.Tensor, box2: torch.Tensor, metric: int = _lib.METRIC_DISCS) -> torch.Tensor:
    """Element-wise overlap of box1[...,5] and box2[...,5] (same shape) -> [...], differentiable."""
    return _Pairwise.apply(box1, box2, metric)


def _allpairs_inputs(ego_box, all_box, mask, metric):
    if ego_box.dim() != 3 or all_box.dim() != 3 or ego_box.shape[-1] != 5 or all_box.shape[-1] != 5:
        raise _lib.TdsError("collision_allpairs: expected ego_box [B,A,5] and all_box [B,N,5]")
    if ego_box.shape[0] != all_box.shape[0] or tuple(mask.shape) != tuple(all_box.shape[:2]):
        raise _lib.TdsError("collision_allpairs: batch / mask shape mismatch")
    if metric not in (_lib.METRIC_DISCS, _lib.METRIC_IOU):
        raise _lib.TdsError(f"collision_allpairs: unknown metric {metric}")
    return _lib.as_f32(ego_box), _lib.as_f32(all_box), _lib.as_u8(mask)


def _allpairs_fwd(ego_box, all_box, mask, metric, ego_is_prefix, out=None):
    """-> (overlap [B,A] float32, argmax [B,A] int32); `out` holds the two buffers (argmax None: not written)."""
    e, a, m = _allpairs_inputs(ego_box, all_box, mask, metric)
    B, A, N = e.shape[0], e.shape[1], a.shape[1]
    if out is None:          # the kernel writes every row
        out = (torch.empty(B, A, dtype=torch.float32, device=e.device), torch.empty(B, A, dtype=torch.int32, device=e.device))
    else:
        _check_out(out[0], (B, A), "collision_allpairs")
    _lib.check(_lib.load().tds_collision_allpairs_fwd(_lib.ptr(e), _lib.ptr(a), _lib.ptr(m), B, A, N, metric,
                                                      1 if ego_is_prefix else 0, _lib.ptr(out[0]), _lib.ptr(out[1]),
                                                      _lib.stream_ptr(e.device)))
    return out


def _allpairs_bwd(ego_box, all_box, mask, metric, ego_is_prefix, argmax, grad, out=None):
    """-> (d ego_box, d all_box); `out` holds the two buffers.  The kernel accumulates into d all_box, which is zeroed
    here first."""
    e, a, m = _allpairs_inputs(ego_box, all_box, mask, metric)
    B, A, N = e.shape[0], e.shape[1], a.shape[1]
    if tuple(argmax.shape) != (B, A):
        raise _lib.TdsError("collision_allpairs: argmax must be [B,A]")
    g = _lib.as_f32(grad)
    ge, ga = (torch.zeros_like(e), torch.zeros_like(a)) if out is None else (out[0], out[1].zero_())
    _lib.check(_lib.load().tds_collision_allpairs_bwd(_lib.ptr(e), _lib.ptr(a), _lib.ptr(m), B, A, N, metric,
                                                      1 if ego_is_prefix else 0, _lib.ptr(g),
                                                      _lib.ptr(_lib.as_i32(argmax)), _lib.ptr(ge), _lib.ptr(ga),
                                                      _lib.stream_ptr(e.device)))
    return ge, ga


class _AllPairs(torch.autograd.Function):
    @staticmethod
    def forward(ctx, ego_box, all_box, mask, metric, ego_is_prefix):
        out, arg = _allpairs_fwd(ego_box, all_box, mask, metric, ego_is_prefix)
        ctx.save_for_backward(ego_box, all_box, mask, arg)
        ctx.meta = (metric, ego_is_prefix)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        ego_box, all_box, mask, arg = ctx.saved_tensors
        return (*_allpairs_bwd(ego_box, all_box, mask, *ctx.meta, arg, grad_out), None, None, None)


def collision_allpairs(ego_box: torch.Tensor, all_box: torch.Tensor, mask: torch.Tensor,
                       metric: int = _lib.METRIC_DISCS, ego_is_prefix: bool = True, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Fused Simulator.compute_collision: ego_box [B,A,5], all_box [B,N,5], mask [B,N] -> [B,A], differentiable.
    `out` (contiguous float32 [B,A]): written directly, no autograd tape."""
    if out is None:
        return _AllPairs.apply(ego_box, all_box, mask, metric, ego_is_prefix)
    return _allpairs_fwd(ego_box, all_box, mask, metric, ego_is_prefix, (out, None))[0]


def _agent_boxes(state, size=None, out=None):
    """state [...,4], size [...,2+] -> boxes [...,5]; without `size`: the camera of every agent, (xy [...,2],
    (sin psi, cos psi) [...,2]).  `out`: the boxes, or the (xy, sincos) pair."""
    if state.shape[-1] != 4 or (size is not None and (size.shape[-1] < 2 or state.shape[:-1] != size.shape[:-1])):
        raise _lib.TdsError("agent_boxes: expected state [...,4] and size [...,2]")
    s = _lib.as_f32(state)
    z = None if size is None else _lib.as_f32(size[..., :2])
    if out is None:
        f32 = dict(dtype=torch.float32, device=s.device)
        out = (torch.empty(s.shape[:-1] + (5,), **f32) if size is not None else
               (torch.empty(s.shape[:-1] + (2,), **f32), torch.empty(s.shape[:-1] + (2,), **f32)))
    box, (xy, sc) = (out, (None, None)) if size is not None else (None, out)
    _lib.check(_lib.load().tds_agent_boxes(_lib.ptr(s), _lib.ptr(z), s.numel() // 4, _lib.ptr(box), _lib.ptr(sc), _lib.ptr(xy),
                                           _lib.stream_ptr(s.device)))
    return out


def _agent_boxes_grad(g, size_cols: int):
    """d boxes [...,5] -> (d state [...,4], d size [...,size_cols])."""
    gs = torch.cat([g[..., 0:2], g[..., 4:5], torch.zeros_like(g[..., 0:1])], dim=-1)
    gz = g[..., 2:4]
    if size_cols > 2:
        gz = torch.cat([gz, g.new_zeros(gz.shape[:-1] + (size_cols - 2,))], dim=-1)
    return gs, gz


class _AgentBoxes(torch.autograd.Function):
    @staticmethod
    def forward(ctx, state, size):
        ctx.size_cols = size.shape[-1]
        return _agent_boxes(state, size)

    @staticmethod
    def backward(ctx, g):
        return _agent_boxes_grad(g, ctx.size_cols)


def agent_boxes(state: torch.Tensor, size: torch.Tensor) -> torch.Tensor:
    """state [...,4] (x, y, psi, v), size [...,2+] (length, width) -> boxes [...,5] (x, y, length, width, psi): the layout of
    compute_collision (simulator.py:1161-1170) in one launch instead of a torch.cat; differentiable."""
    return _AgentBoxes.apply(state, size)


def egocentric_cameras(state: torch.Tensor):
    """state [...,4] -> (xy [...,2] contiguous, (sin psi, cos psi) [...,2]): the camera of every agent in one launch, the
    heading evaluated like every other heading of the path (float64, rounded) - render_egocentric, simulator.py:961,
    1017.  Not differentiable."""
    return _agent_boxes(state)


def heading_sincos(state: torch.Tensor) -> torch.Tensor:
    return egocentric_cameras(state)[1]


# ------------------------------------------------------------------------------------ traffic lights
def traffic_light_violation(agent_box: torch.Tensor, tl_corners: torch.Tensor, tl_state: torch.Tensor, red_state: int,
                            rear_factor: float = 0.1, present: Optional[torch.Tensor] = None) -> torch.Tensor:
    """agent_box [B,A,5], tl_corners [B,L,4,2], tl_state [B,L] -> bool [B,A]
    (TrafficLightControl.compute_violation, traffic_controls.py:152-178; not differentiable, as the reference)."""
    lib = _lib.load()
    box = _lib.as_f32(agent_box)
    if box.dim() != 3 or box.shape[-1] != 5:
        raise _lib.TdsError("traffic_light_violation: agent_box must be [B,A,5]")
    B, A = box.shape[0], box.shape[1]
    L = tl_corners.shape[1]
    if tl_corners.shape[0] != B or tuple(tl_corners.shape[2:]) != (4, 2) or tuple(tl_state.shape) != (B, L):
        raise _lib.TdsError("traffic_light_violation: tl_corners must be [B,L,4,2] and tl_state [B,L]")
    out = torch.zeros(B, A, dtype=torch.uint8, device=box.device)
    cor = _lib.as_f32(tl_corners) if L > 0 else None
    st = _lib.as_i32(tl_state.to(box.device)) if L > 0 else None
    p = None if present is None else _lib.as_u8(present)
    _lib.check(lib.tds_traffic_light_violation(_lib.ptr(box), _lib.ptr(cor), _lib.ptr(st), _lib.ptr(p), B, A, L,
                                               int(red_state), float(rear_factor), _lib.ptr(out), _lib.stream_ptr(box.device)))
    return out.view(torch.bool)


def _agents_relative_shape(absolute, n_agents, exclude_self, what="agents_relative"):
    """-> (B, A, N, M): the output is [B,A,M,6].  With absolute [B,A,N,6] (per origin) `n_agents` is not used."""
    if absolute.dim() not in (3, 4) or absolute.shape[-1] != 6:
        raise _lib.TdsError(f"{what}: absolute must be [B,N,6] or [B,A,N,6]")
    B, N = absolute.shape[0], absolute.shape[-2]
    A = absolute.shape[1] if absolute.dim() == 4 else (N if n_agents is None else int(n_agents))
    if not 0 <= A <= N:
        raise _lib.TdsError(f"{what}: n_agents must be in [0, N]")
    return B, A, N, (max(N - 1, 0) if exclude_self else N)


def _agents_relative_fwd(absolute, n_agents, exclude_self):
    B, A, N, M = _agents_relative_shape(absolute, n_agents, exclude_self)
    a = _lib.as_f32(absolute)
    out = torch.empty(B, A, M, 6, dtype=torch.float32, device=a.device)
    _lib.check(_lib.load().tds_agents_relative(_lib.ptr(a), B, A, N, 1 if exclude_self else 0, 1 if a.dim() == 4 else 0,
                                               _lib.ptr(out), _lib.stream_ptr(a.device)))
    return out


def _agents_relative_bwd(absolute, n_agents, exclude_self, grad):
    """-> d absolute (float32, the shape of `absolute`); every element is written by the kernel."""
    B, A, N, M = _agents_relative_shape(absolute, n_agents, exclude_self)
    if tuple(grad.shape) != (B, A, M, 6):
        raise _lib.TdsError(f"agents_relative: the gradient must be [B,A,M,6] = {[B, A, M, 6]}")
    a, g = _lib.as_f32(absolute), _lib.as_f32(grad)
    ga = torch.empty_like(a)
    _lib.check(_lib.load().tds_agents_relative_bwd(_lib.ptr(a), _lib.ptr(g), B, A, N, 1 if exclude_self else 0,
                                                   1 if a.dim() == 4 else 0, _lib.ptr(ga), _lib.stream_ptr(a.device)))
    return ga


class _AgentsRelative(torch.autograd.Function):
    @staticmethod
    def forward(ctx, absolute, n_agents, exclude_self):
        ctx.save_for_backward(absolute)
        ctx.meta = (n_agents, exclude_self)
        return _agents_relative_fwd(absolute, n_agents, exclude_self)

    @staticmethod
    def backward(ctx, grad_out):
        return _agents_relative_bwd(*ctx.saved_tensors, *ctx.meta, grad_out), None, None


def agents_relative(absolute: torch.Tensor, n_agents: Optional[int] = None, exclude_self: bool = True) -> torch.Tensor:
    """absolute [B,N,6] (x, y, psi, length, width, present) -> [B,A,N(-1),6]: every agent in the frame of each of the
    first `n_agents` agents (Simulator.get_all_agents_relative, simulator.py:748-781).  With absolute [B,A,N,6] (what
    each agent perceives, get_noisy_all_agents_absolute) row i is relative to its own entry [b,i,i]
    (get_noisy_all_agents_relative, simulator.py:784-821).  The self entry is removed on the device without the
    reference's synchronising boolean-mask index.  Differentiable in `absolute`, as the reference's torch arithmetic:
    the backward kernel (tds_agents_relative_bwd) recomputes the pairs from `absolute` and needs no saved output."""
    return _AgentsRelative.apply(absolute, n_agents, exclude_self)


def _nearest_shape(absolute, k, n_agents):
    """-> (B, A, N, k): the outputs are [B,A,k,6] and [B,A,k]."""
    B, A, N, _ = _agents_relative_shape(absolute, n_agents, False, "nearest_agents_relative")
    try:
        k = operator.index(k)
    except TypeError:
        k = 0
    if not 1 <= k <= 64:
        raise _lib.TdsError("nearest_agents_relative: k must be an integer in [1, 64]")
    return B, A, N, k


def _nearest_r2(max_distance, what="nearest_agents_relative"):
    """float32(max_distance ** 2), squared in double precision and rounded once (to +inf past the float32 range)."""
    if not max_distance >= 0:
        raise _lib.TdsError(f"{what}: max_distance must be >= 0")
    return ctypes.c_float(float(max_distance) * float(max_distance)).value


def _nearest_fwd(absolute, k, n_agents, max_distance):
    B, A, N, k = _nearest_shape(absolute, k, n_agents)
    r2 = _nearest_r2(max_distance)
    a = _lib.as_f32(absolute)
    out = torch.empty(B, A, k, 6, dtype=torch.float32, device=a.device)
    idx = torch.empty(B, A, k, dtype=torch.int64, device=a.device)
    _lib.check(_lib.load().tds_nearest_agents_relative(_lib.ptr(a), B, A, N, k, 1 if a.dim() == 4 else 0, r2,
                                                       _lib.ptr(out), _lib.ptr(idx), _lib.stream_ptr(a.device)))
    return out, idx


def _nearest_bwd(absolute, k, n_agents, idx, grad):
    """-> d absolute (float32, the shape of `absolute`); every element is written by the kernel."""
    B, A, N, k = _nearest_shape(absolute, k, n_agents)
    if tuple(idx.shape) != (B, A, k) or idx.dtype != torch.int64:
        raise _lib.TdsError(f"nearest_agents_relative: idx must be int64 [B,A,k] = {[B, A, k]}")
    if tuple(grad.shape) != (B, A, k, 6):
        raise _lib.TdsError(f"nearest_agents_relative: the gradient must be [B,A,k,6] = {[B, A, k, 6]}")
    a, g, i = _lib.as_f32(absolute), _lib.as_f32(grad), idx.detach().contiguous()
    ga = torch.empty_like(a)
    _lib.check(_lib.load().tds_nearest_agents_relative_bwd(_lib.ptr(a), _lib.ptr(i), _lib.ptr(g), B, A, N, k,
                                                           1 if a.dim() == 4 else 0, _lib.ptr(ga), _lib.stream_ptr(a.device)))
    return ga


class _NearestAgentsRelative(torch.autograd.Function):
    @staticmethod
    def forward(ctx, absolute, k, n_agents, max_distance):
        out, idx = _nearest_fwd(absolute, k, n_agents, max_distance)
        ctx.save_for_backward(absolute, idx)
        ctx.meta = (k, n_agents)
        ctx.mark_non_differentiable(idx)
        return out, idx

    @staticmethod
    def backward(ctx, grad_out, grad_idx):
        absolute, idx = ctx.saved_tensors
        return _nearest_bwd(absolute, *ctx.meta, idx, grad_out), None, None, None


def nearest_agents_relative(absolute: torch.Tensor, k: int, n_agents: Optional[int] = None,
                            max_distance: float = math.inf) -> Tuple[torch.Tensor, torch.Tensor]:
    """The k nearest agents of every origin in its frame: -> (relative [B,A,k,6], idx [B,A,k] int64).  `absolute` and
    `n_agents` as for `agents_relative` (shared origins [B,N,6] or per origin [B,A,N,6]), 1 <= k <= 64.
    Agent j != i is eligible for origin i iff it is present and its float32 squared distance
    (x_j - x_i)^2 + (y_j - y_i)^2 (no FMA) is <= float32(max_distance ** 2); a NaN position is never eligible.  The
    eligible agents are sorted by (squared distance, j); slot s of row i holds exactly
    `agents_relative(absolute, n_agents, exclude_self=False)[b, i, j]` of the s-th one and idx its j.  Slots past the
    eligible agents are zero with idx -1.  Differentiable in `absolute` through the filled slots, as the matching
    entries of `agents_relative` (the selection itself is piecewise constant).  One launch each way, no host
    synchronisation, and nothing of size [B,A,N] is formed: the output is 24 k bytes per origin."""
    return _NearestAgentsRelative.apply(absolute, k, n_agents, max_distance)


def sensing_noise(all_state: torch.Tensor, n_agents: int, eps: Optional[torch.Tensor] = None) -> torch.Tensor:
    """all_state [B,N,4] -> [B,A,N,4]: the states the first `n_agents` agents perceive, with noise growing with the
    distance (StandardSensingObservationNoise.get_noisy_state, observation_noise.py:74-89).  `eps` [B,A,N,4] are the
    standard normal deviates (drawn on the device when omitted)."""
    lib = _lib.load()
    s = _lib.as_f32(all_state)
    if s.dim() != 3 or s.shape[-1] != 4:
        raise _lib.TdsError("sensing_noise: all_state must be [B,N,4]")
    B, N = s.shape[0], s.shape[1]
    A = int(n_agents)
    if eps is None:
        eps = torch.randn(B, A, N, 4, dtype=torch.float32, device=s.device)
    eps = _lib.as_f32(eps)
    if tuple(eps.shape) != (B, A, N, 4):
        raise _lib.TdsError("sensing_noise: eps must be [B,A,N,4]")
    out = torch.empty(B, A, N, 4, dtype=torch.float32, device=s.device)
    _lib.check(lib.tds_sensing_noise(_lib.ptr(s), _lib.ptr(eps), B, A, N, _lib.ptr(out), _lib.stream_ptr(s.device)))
    return out


def sensing_occlusion(all_state: torch.Tensor, all_size: torch.Tensor, base_mask: torch.Tensor, n_agents: int) -> torch.Tensor:
    """all_state [B,N,4], all_size [B,N,2], base_mask [B,N] -> bool [B,A,N]: present and in the line of sight of each of
    the first `n_agents` agents (StandardSensingObservationNoise.get_noisy_present_mask, observation_noise.py:91-132)."""
    lib = _lib.load()
    s, z, m = _lib.as_f32(all_state), _lib.as_f32(all_size), _lib.as_u8(base_mask)
    B, N = s.shape[0], s.shape[1]
    if s.dim() != 3 or s.shape[-1] != 4 or tuple(z.shape) != (B, N, 2) or tuple(m.shape) != (B, N):
        raise _lib.TdsError("sensing_occlusion: expected all_state [B,N,4], all_size [B,N,2], base_mask [B,N]")
    A = int(n_agents)
    out = torch.empty(B, A, N, dtype=torch.uint8, device=s.device)
    _lib.check(lib.tds_sensing_occlusion(_lib.ptr(s), _lib.ptr(z), _lib.ptr(m), B, A, N, _lib.ptr(out), _lib.stream_ptr(s.device)))
    return out.view(torch.bool)


def infraction_metrics(collision: torch.Tensor, offroad: torch.Tensor, present: Optional[torch.Tensor] = None,
                       acc: Optional[torch.Tensor] = None) -> torch.Tensor:
    """[6] float64, accumulated into `acc` when given: collision sum, offroad sum, colliding agents, offroad agents,
    present agents, agent slots (distributed.METRIC_NAMES) - the vector a multi-GPU job all-reduces.  One launch."""
    lib = _lib.load()
    c, o = _lib.as_f32(collision), _lib.as_f32(offroad)
    if c.shape != o.shape:
        raise _lib.TdsError("infraction_metrics: collision and offroad must have the same shape")
    p = None if present is None else _lib.as_u8(present)
    if p is not None and p.shape != c.shape:
        raise _lib.TdsError("infraction_metrics: present must have the shape of collision")
    if acc is None:
        acc = torch.zeros(6, dtype=torch.float64, device=c.device)
    elif acc.dtype != torch.float64 or acc.numel() != 6 or not acc.is_contiguous():
        raise _lib.TdsError("infraction_metrics: acc must be a contiguous float64 tensor of 6 elements")
    _lib.check(lib.tds_infraction_metrics(_lib.ptr(c), _lib.ptr(o), _lib.ptr(p), c.numel(), _lib.ptr(acc), _lib.stream_ptr(c.device)))
    return acc


# ------------------------------------------------------------------------------------ offroad
def _offroad_inputs(state, lenwid, present):
    if state.dim() != 3 or state.shape[-1] != 4:
        raise _lib.TdsError("offroad: expected state [B,A,4]")
    if tuple(lenwid.shape) != (state.shape[0], state.shape[1], 2):
        raise _lib.TdsError("offroad: expected lenwid [B,A,2] or [B,2]")
    if present is not None and tuple(present.shape) != tuple(state.shape[:2]):
        raise _lib.TdsError("offroad: expected present [B,A]")
    return _lib.as_f32(state), _lib.as_f32(lenwid), None if present is None else _lib.as_u8(present)


def _offroad_fwd(state, lenwid, present, mapset, threshold, out=None):
    """-> (offroad [B,A] float32, face [B,A,4] int32: the face each corner was measured to, -1 for none); `out` holds
    the two buffers (face None: not written)."""
    s, lw, p = _offroad_inputs(state, lenwid, present)
    B, A = s.shape[0], s.shape[1]
    if out is None:          # the kernel writes every agent
        out = (torch.empty(B, A, dtype=torch.float32, device=s.device), torch.empty(B, A, 4, dtype=torch.int32, device=s.device))
    else:
        _check_out(out[0], (B, A), "offroad")
    handles, n_maps = mapset.handles(s.device)
    _lib.check(_lib.load().tds_offroad_fwd(handles, n_maps, _lib.ptr(mapset.env_map_on(s.device)), _lib.ptr(s), _lib.ptr(lw),
                                           _lib.ptr(p), B, A, float(threshold), _lib.ptr(out[0]), _lib.ptr(out[1]),
                                           _lib.stream_ptr(s.device)))
    return out


def _offroad_bwd(state, lenwid, present, mapset, threshold, face, grad, out=None):
    """-> (d state, d lenwid); `out` holds the two buffers, None for a gradient that is not wanted."""
    s, lw, p = _offroad_inputs(state, lenwid, present)
    g = _lib.as_f32(grad)
    gs, gl = (torch.zeros_like(s), torch.zeros_like(lw)) if out is None else out
    handles, n_maps = mapset.handles(s.device)
    _lib.check(_lib.load().tds_offroad_bwd(handles, n_maps, _lib.ptr(mapset.env_map_on(s.device)), _lib.ptr(s), _lib.ptr(lw),
                                           _lib.ptr(p), s.shape[0], s.shape[1], float(threshold), _lib.ptr(face), _lib.ptr(g),
                                           _lib.ptr(gs), _lib.ptr(gl), _lib.stream_ptr(s.device)))
    return gs, gl


class _Offroad(torch.autograd.Function):
    @staticmethod
    def forward(ctx, state, lenwid, present, mapset, threshold):
        out, face = _offroad_fwd(state, lenwid, present, mapset, threshold)
        ctx.save_for_backward(state, lenwid, present, face)
        ctx.meta = (mapset, threshold)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        state, lenwid, present, face = ctx.saved_tensors
        return (*_offroad_bwd(state, lenwid, present, *ctx.meta, face, grad_out), None, None, None)


def offroad(state: torch.Tensor, lenwid: torch.Tensor, mapset: MapSet, threshold: float = 0.0,
            present: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """state [B,A,4], lenwid [B,A,2] or [B,2], present [B,A] -> [B,A] sum over corners of thresholded squared distance
    to the map.  `out` (contiguous float32 [B,A]): written directly, no autograd tape."""
    if lenwid.dim() == 2 and state.dim() == 3:
        lenwid = lenwid.unsqueeze(-2).expand(lenwid.shape[0], state.shape[1], lenwid.shape[1])
    if out is None:
        return _Offroad.apply(state, lenwid, present, mapset, threshold)
    return _offroad_fwd(state, lenwid, present, mapset, threshold, (out, None))[0]


# ------------------------------------------------------------------------------------ map observations
def _map_segments_shape(state, mapset, k):
    """-> (B, A, k): the outputs are [B,A,k,4] and [B,A,k]."""
    if state.dim() != 3 or state.shape[-1] != 4:
        raise _lib.TdsError("nearest_map_segments: expected state [B,A,4]")
    try:
        k = operator.index(k)
    except TypeError:
        k = 0
    if not 1 <= k <= 256:
        raise _lib.TdsError("nearest_map_segments: k must be an integer in [1, 256]")
    if mapset.env_map is not None and tuple(mapset.env_map.shape) != (state.shape[0],):
        raise _lib.TdsError("nearest_map_segments: the map set's env_map must be [B]")
    return state.shape[0], state.shape[1], k


def _map_segments_fwd(state, mapset, k, max_distance):
    """-> (rel [B,A,k,4] float32, kind [B,A,k] int64, idx [B,A,k] int64)."""
    B, A, k = _map_segments_shape(state, mapset, k)
    r2 = _nearest_r2(max_distance, "nearest_map_segments")
    s = _lib.as_f32(state)
    rel = torch.empty(B, A, k, 4, dtype=torch.float32, device=s.device)
    kind = torch.empty(B, A, k, dtype=torch.int64, device=s.device)
    idx = torch.empty(B, A, k, dtype=torch.int64, device=s.device)
    handles, n_maps = mapset.handles(s.device)
    _lib.check(_lib.load().tds_nearest_map_segments(handles, n_maps, _lib.ptr(mapset.env_map_on(s.device)), _lib.ptr(s), B, A,
                                                    k, r2, _lib.ptr(rel), _lib.ptr(kind), _lib.ptr(idx),
                                                    _lib.stream_ptr(s.device)))
    return rel, kind, idx


def _map_segments_bwd(state, mapset, k, idx, grad):
    """-> d state [B,A,4] float32 (v gets 0); every element is written by the kernel."""
    B, A, k = _map_segments_shape(state, mapset, k)
    if tuple(idx.shape) != (B, A, k) or idx.dtype != torch.int64:
        raise _lib.TdsError(f"nearest_map_segments: idx must be int64 [B,A,k] = {[B, A, k]}")
    if tuple(grad.shape) != (B, A, k, 4):
        raise _lib.TdsError(f"nearest_map_segments: the gradient must be [B,A,k,4] = {[B, A, k, 4]}")
    s, g, i = _lib.as_f32(state), _lib.as_f32(grad), idx.detach().contiguous()
    gs = torch.empty(B, A, 4, dtype=torch.float32, device=s.device)
    handles, n_maps = mapset.handles(s.device)
    _lib.check(_lib.load().tds_nearest_map_segments_bwd(handles, n_maps, _lib.ptr(mapset.env_map_on(s.device)), _lib.ptr(s),
                                                        _lib.ptr(i), _lib.ptr(g), B, A, k, _lib.ptr(gs),
                                                        _lib.stream_ptr(s.device)))
    return gs


class _NearestMapSegments(torch.autograd.Function):
    @staticmethod
    def forward(ctx, state, mapset, k, max_distance):
        rel, kind, idx = _map_segments_fwd(state, mapset, k, max_distance)
        ctx.save_for_backward(state, idx)
        ctx.meta = (mapset, k)
        ctx.mark_non_differentiable(kind, idx)
        return rel, kind, idx

    @staticmethod
    def backward(ctx, grad_rel, grad_kind, grad_idx):
        state, idx = ctx.saved_tensors
        mapset, k = ctx.meta
        return _map_segments_bwd(state, mapset, k, idx, grad_rel), None, None, None


def nearest_map_segments(state: torch.Tensor, mapset: MapSet, k: int,
                         max_distance: float = math.inf) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """The k nearest lane-marking segments of every agent, in its frame: state [B,A,4] (x, y, psi, v) ->
    (rel [B,A,k,4] float32, kind [B,A,k] int64, idx [B,A,k] int64), 1 <= k <= 256; `mapset.maps[env_map[b]]` is the map
    of environment b.

    Segment s of a map is the s-th strip of four faces (a,b,c),(b,c,d),(c,d,e),(d,e,f) of one class in face order
    (what the reference's line_segments_to_mesh draws for a lane-marking segment [p0, p1] = [c, d]); its kind is the
    strip's palette class (`palette.class_names()[kind]`); see `StaticMap.marking_segments`.  The key of segment
    (p0, p1) for agent (x, y) is the float32 squared distance from the agent to the segment, every operation rounded on
    its own: e = p1 - p0, w = (x, y) - p0, t = clamp((w . e) / |e|^2, 0, 1) (0 for |e| = 0), key = |w - t e|^2.  A
    segment is eligible iff key <= float32(max_distance ** 2); a NaN key never is, and an agent whose x or y is not finite
    has no eligible segment.  The eligible segments are ordered by (key, s).  Slot j holds both endpoints in the agent's
    frame, (rx0, ry0, rx1, ry1), with the position arithmetic of `agents_relative`, kind its class and idx its s.
    Leftover slots are zero with kind and idx -1.

    Differentiable in the agent's (x, y, psi) through the filled slots (the map is constant and the selection piecewise
    constant; v gets 0).  One launch each way, no host synchronisation: both directions can be captured in a CUDA graph."""
    return _NearestMapSegments.apply(state, mapset, k, max_distance)


def _range_scan_shape(absolute, n_rays, n_agents, mapset):
    """-> (B, A, N, R): the outputs are [B,A,R]."""
    if absolute.dim() != 3 or absolute.shape[-1] != 6:
        raise _lib.TdsError("range_scan: absolute must be [B,N,6]")
    B, A, N, _ = _agents_relative_shape(absolute, n_agents, False, "range_scan")
    try:
        R = operator.index(n_rays)
    except TypeError:
        R = 0
    if not 1 <= R <= 256:
        raise _lib.TdsError("range_scan: n_rays must be an integer in [1, 256]")
    if mapset is not None and mapset.env_map is not None and tuple(mapset.env_map.shape) != (B,):
        raise _lib.TdsError("range_scan: the map set's env_map must be [B]")
    return B, A, N, R


def _range_scan_maps(mapset, device):
    """(handles, n_maps, env_map) of the map set, (None, 0, None) without one."""
    if mapset is None:
        return None, 0, None
    handles, n_maps = mapset.handles(device)
    return handles, n_maps, mapset.env_map_on(device)


def _range_scan_fwd(absolute, n_rays, n_agents, max_range, mapset):
    """-> (dist [B,A,R] float32, kind [B,A,R] int64, idx [B,A,R] int64)."""
    B, A, N, R = _range_scan_shape(absolute, n_rays, n_agents, mapset)
    try:
        r = ctypes.c_float(float(max_range)).value
    except TypeError:
        r = math.nan
    if not (math.isfinite(r) and r > 0):
        raise _lib.TdsError("range_scan: max_range must be finite and > 0 in float32")
    a = _lib.as_f32(absolute)
    dist = torch.empty(B, A, R, dtype=torch.float32, device=a.device)
    kind = torch.empty(B, A, R, dtype=torch.int64, device=a.device)
    idx = torch.empty(B, A, R, dtype=torch.int64, device=a.device)
    handles, n_maps, env_map = _range_scan_maps(mapset, a.device)
    _lib.check(_lib.load().tds_range_scan(handles, n_maps, _lib.ptr(env_map), _lib.ptr(a), B, A, N, R, r, _lib.ptr(dist),
                                          _lib.ptr(kind), _lib.ptr(idx), _lib.stream_ptr(a.device)))
    return dist, kind, idx


def _range_scan_bwd(absolute, n_rays, n_agents, mapset, kind, idx, grad):
    """-> d absolute [B,N,6] float32 (the present column gets 0); every element is written by the kernel."""
    B, A, N, R = _range_scan_shape(absolute, n_rays, n_agents, mapset)
    for name, t in (("kind", kind), ("idx", idx)):
        if tuple(t.shape) != (B, A, R) or t.dtype != torch.int64:
            raise _lib.TdsError(f"range_scan: {name} must be int64 [B,A,R] = {[B, A, R]}")
    if tuple(grad.shape) != (B, A, R):
        raise _lib.TdsError(f"range_scan: the gradient must be [B,A,R] = {[B, A, R]}")
    a, g = _lib.as_f32(absolute), _lib.as_f32(grad)
    k, i = kind.detach().contiguous(), idx.detach().contiguous()
    ga = torch.empty_like(a)
    handles, n_maps, env_map = _range_scan_maps(mapset, a.device)
    _lib.check(_lib.load().tds_range_scan_bwd(handles, n_maps, _lib.ptr(env_map), _lib.ptr(a), _lib.ptr(k), _lib.ptr(i),
                                              _lib.ptr(g), B, A, N, R, _lib.ptr(ga), _lib.stream_ptr(a.device)))
    return ga


class _RangeScan(torch.autograd.Function):
    @staticmethod
    def forward(ctx, absolute, n_rays, n_agents, max_range, mapset):
        dist, kind, idx = _range_scan_fwd(absolute, n_rays, n_agents, max_range, mapset)
        ctx.save_for_backward(absolute, kind, idx)
        ctx.meta = (n_rays, n_agents, mapset)
        ctx.mark_non_differentiable(kind, idx)
        return dist, kind, idx

    @staticmethod
    def backward(ctx, grad_dist, grad_kind, grad_idx):
        absolute, kind, idx = ctx.saved_tensors
        n_rays, n_agents, mapset = ctx.meta
        return _range_scan_bwd(absolute, n_rays, n_agents, mapset, kind, idx, grad_dist), None, None, None, None


def range_scan(absolute: torch.Tensor, n_rays: int, n_agents: Optional[int] = None, max_range: float = 50.0,
               mapset: Optional[MapSet] = None) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """The distance along `n_rays` rays of every origin agent to the first agent box or lane marking:
    absolute [B,N,6] (x, y, psi, length, width, present; get_all_agents_absolute) -> (dist [B,A,R] float32,
    kind [B,A,R] int64, idx [B,A,R] int64).  The origins are the first A = `n_agents` rows (default N), each computed
    whatever its own present flag; 1 <= R = n_rays <= 256; `max_range` is finite and > 0 and used as float32(max_range).
    With `mapset` (`mapset.maps[env_map[b]]` the map of environment b) the lane markings are candidates too.

    Ray r of origin i has the unit vector u_r = (cos, sin)(2 pi r / R) in the agent's frame (the frame of
    `agents_relative`), evaluated in double with sincospi(2r/R) and rounded to float32, so rays at quarter turns are
    exact axis vectors.  With (s, c) = sincos(psi_i) (double, rounded), the world direction is d = (c ux - s uy,
    s ux + c uy) and the origin o = (x_i, y_i).  The candidates are segments: edge k of the box of every agent j != i of
    the environment with present_j != 0, from corner k to corner (k + 1) % 4 (the corners of `offroad`, in the order of
    box2corners_th), code 4 j + k; with a map, every lane-marking segment s of `StaticMap.marking_segments`, code
    4 N + s.  The hit test is float32 with every operation rounded on its own and IEEE division: e = p1 - p0, w = p0 - o,
    den = dx ey - dy ex; den == 0 is no hit; else t = (wx ey - wy ex) / den, u = (wx dy - wy dx) / den, and it is a hit
    iff 0 <= u <= 1 and 0 <= t <= float32(max_range).  A NaN never hits; a t of -0 counts as +0.  The winner is the
    smallest word (bits(t) << 32) | code: the nearest hit, on equal t the smaller code.  dist is its t, or
    float32(max_range) without a hit; kind is 0 for an agent edge, 1 for a marking, -1 for none; idx is the agent row j,
    the segment index s, or -1.  An origin whose x, y or psi is not finite hits nothing.

    dist is differentiable in `absolute`: the origin's x, y, psi and, for an agent hit, the hit agent's x, y, psi, length
    and width (the map is constant, the present column gets 0, the selection is piecewise constant).  A ray without a
    hit contributes nothing, not even a NaN upstream value.  One launch each way, no host synchronisation: both
    directions can be captured in a CUDA graph.  Output per origin: 20 bytes per ray."""
    return _RangeScan.apply(absolute, n_rays, n_agents, max_range, mapset)


# ------------------------------------------------------------------------------------ time to collision
def _ttc_shape(state, size, present, n_agents, horizon):
    """-> (B, A, N, H): the outputs are [B,A]; H = float32(horizon), finite and > 0."""
    if state.dim() != 3 or state.shape[-1] != 4:
        raise _lib.TdsError("time_to_collision: state must be [B,N,4]")
    B, N = state.shape[0], state.shape[1]
    if tuple(size.shape) != (B, N, 2):
        raise _lib.TdsError(f"time_to_collision: size must be [B,N,2] = {[B, N, 2]}")
    if tuple(present.shape) != (B, N):
        raise _lib.TdsError(f"time_to_collision: present must be [B,N] = {[B, N]}")
    try:
        A = N if n_agents is None else operator.index(n_agents)
    except TypeError:
        A = -1
    if not 0 <= A <= N:
        raise _lib.TdsError("time_to_collision: n_agents must be an integer in [0, N]")
    try:
        H = ctypes.c_float(float(horizon)).value
    except TypeError:
        H = math.nan
    if not (math.isfinite(H) and H > 0):
        raise _lib.TdsError("time_to_collision: horizon must be finite and > 0 in float32")
    return B, A, N, H


def _time_to_collision_fwd(state, size, present, n_agents, horizon):
    """-> (ttc [B,A] float32, idx [B,A] int64); every element is written by the kernel."""
    B, A, N, H = _ttc_shape(state, size, present, n_agents, horizon)
    s, z, p = _lib.as_f32(state), _lib.as_f32(size), _lib.as_u8(present)
    ttc = torch.empty(B, A, dtype=torch.float32, device=s.device)
    idx = torch.empty(B, A, dtype=torch.int64, device=s.device)
    _lib.check(_lib.load().tds_time_to_collision(_lib.ptr(s), _lib.ptr(z), _lib.ptr(p), B, A, N, H, _lib.ptr(ttc),
                                                 _lib.ptr(idx), _lib.stream_ptr(s.device)))
    return ttc, idx


def _time_to_collision_bwd(state, size, present, n_agents, horizon, idx, grad):
    """-> (d state [B,N,4], d size [B,N,2]) float32; every element is written by the kernel."""
    B, A, N, H = _ttc_shape(state, size, present, n_agents, horizon)
    if tuple(idx.shape) != (B, A) or idx.dtype != torch.int64:
        raise _lib.TdsError(f"time_to_collision: idx must be int64 [B,A] = {[B, A]}")
    if tuple(grad.shape) != (B, A):
        raise _lib.TdsError(f"time_to_collision: the gradient must be [B,A] = {[B, A]}")
    s, z, p = _lib.as_f32(state), _lib.as_f32(size), _lib.as_u8(present)
    g, i = _lib.as_f32(grad), idx.detach().contiguous()
    gs, gz = torch.empty_like(s), torch.empty_like(z)
    _lib.check(_lib.load().tds_time_to_collision_bwd(_lib.ptr(s), _lib.ptr(z), _lib.ptr(p), B, A, N, H, _lib.ptr(g),
                                                     _lib.ptr(i), _lib.ptr(gs), _lib.ptr(gz), _lib.stream_ptr(s.device)))
    return gs, gz


class _TimeToCollision(torch.autograd.Function):
    @staticmethod
    def forward(ctx, state, size, present, horizon, n_agents):
        ttc, idx = _time_to_collision_fwd(state, size, present, n_agents, horizon)
        ctx.save_for_backward(state, size, present, idx)
        ctx.meta = (n_agents, horizon)
        ctx.mark_non_differentiable(idx)
        return ttc, idx

    @staticmethod
    def backward(ctx, grad_ttc, grad_idx):
        state, size, present, idx = ctx.saved_tensors
        n_agents, horizon = ctx.meta
        gs, gz = _time_to_collision_bwd(state, size, present, n_agents, horizon, idx, grad_ttc)
        return gs, gz, None, None, None


def time_to_collision(state: torch.Tensor, size: torch.Tensor, present: torch.Tensor, horizon: float = 5.0,
                      n_agents: Optional[int] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Time to collision (TTC): the first contact of every origin agent under constant velocity, all pairs ->
    (ttc [B,A] float32, idx [B,A] int64).

    Inputs: state [B,N,4] (x, y, psi, v); size [B,N,2] (length, width); present [B,N] bool; n_agents = A <= N (default
    N): rows 0..A-1 are the origins, all N rows are candidates, so NPCs take part, as in compute_collision; horizon H in
    seconds, finite and > 0, used as float32(horizon).

    Every agent keeps its heading and its speed: box j at time t has centre (x_j + t * vx_j, y_j + t * vy_j), with
    vx_j = v_j * c_j, vy_j = v_j * s_j, and (s_j, c_j) = sincos_cr(psi_j) (double precision, rounded to float32), which
    is the heading evaluation the whole path uses.  This is a definition, not the kinematic model's prediction: the
    bicycle's slip angle is ignored, as every TTC metric does.

    Pair (i, j), for j != i with both present, uses float32 arithmetic.  Every operation is rounded on its own (the
    library is -fmad=false) and divisions are IEEE.  The four separating axes are taken in this order:
    1. u_i = (c_i, s_i),  2. u_i⊥ = (-s_i, c_i),  3. u_j,  4. u_j⊥.
    For axis n = (nx, ny): d0 = nx * (x_j - x_i) + ny * (y_j - y_i), s = nx * (vx_j - vx_i) + ny * (vy_j - vy_i),
    R = h_i + h_j.  A box's half-extent on its own axes is exactly 0.5 * length or 0.5 * width.  On the other box's
    axes it is |n·u| * 0.5 * length + |n·u⊥| * 0.5 * width.
    Entry and exit times per axis: if s != 0, ta = (-R - d0) / s and tb = (R - d0) / s, entry min(ta, tb) and exit
    max(ta, tb); if s == 0, entry is -inf and exit +inf when |d0| <= R, otherwise the pair never touches.
    T_in is the maximum of the four entries and T_out the minimum of the four exits.  The pair touches within the
    horizon iff max(T_in, 0) <= min(T_out, H).  Its time is T_in > 0 ? T_in : +0.0 (no negative zero, so keys order by
    their bits).  Boxes that overlap at t = 0 give 0.  A pair whose time is NaN never counts.

    ttc and idx are the minimum over j of the pair time, ties going to the smaller j (the key is bits(t) << 32 | j).
    If no pair touches, or origin i is absent: ttc = +inf and idx = -1.

    ttc is differentiable in the (x, y, psi, v) and (length, width) of the origin and of agent idx, where
    0 < ttc < inf.  There ttc = -(d0 + sgn(s) R) / s on the first axis, in the order above, whose entry equals T_in,
    with dt/dd0 = -1/s, dt/dR = -1/|s| and dt/ds = -t/s, chained through d0, s and R to both agents (the derivative of
    |x| is sgn(x), 0 at 0).  Rows with ttc == 0 or idx == -1 are skipped by a branch, so an inf or NaN upstream value
    there never reaches a gradient.  One launch each way, no host synchronisation: both directions can be captured in
    a CUDA graph."""
    return _TimeToCollision.apply(state, size, present, horizon, n_agents)


# ------------------------------------------------------------------------------------ raster
def raster_birdview(mapset: MapSet, palette: "_lib.Palette", cam_xy: torch.Tensor, cam_sc: torch.Tensor,
                    agent_state: Optional[torch.Tensor], agent_size: Optional[torch.Tensor],
                    agent_type: Optional[torch.Tensor], present: Optional[torch.Tensor],
                    tl_corners: Optional[torch.Tensor], tl_state: Optional[torch.Tensor],
                    rect_corners: Optional[torch.Tensor], rect_class: Optional[torch.Tensor],
                    res: int, fov: float, out: Optional[torch.Tensor] = None,
                    workspace: Optional[torch.Tensor] = None, cam_tris: Optional[torch.Tensor] = None,
                    cam_tri_class: Optional[torch.Tensor] = None, image_format: int = _lib.IMAGE_F32,
                    agent_class: Optional[torch.Tensor] = None) -> torch.Tensor:
    """cam_xy, cam_sc [B,Nc,2] -> images [B,Nc,3,res,res] float32 in [0,255] (not differentiable, like
    the cv2 backend).  present is [B,N] or [B,Nc,N]; cam_tris [B,Nc,Tc,3,2] + cam_tri_class [B,Nc,Tc] are
    triangles seen by one camera each (waypoint discs).  image_format: IMAGE_F32 (the reference's dtype),
    IMAGE_U8 (the same values as uint8 [B,Nc,3,res,res]) or IMAGE_RANK (uint8 [B,Nc,res,res] draw ranks, see
    `raster_rank_table`).  agent_class [B,Nc,N] uint8: palette class of each agent's rectangle per camera (custom colours)."""
    lib = _lib.load()
    dev = cam_xy.device
    cxy, csc = _lib.as_f32(cam_xy), _lib.as_f32(cam_sc)
    B, Nc = cxy.shape[0], cxy.shape[1]
    N = 0 if agent_state is None else agent_state.shape[-2]
    L = 0 if tl_corners is None else tl_corners.shape[1]
    R = 0 if rect_corners is None else rect_corners.shape[1]
    ast = None if N == 0 else _lib.as_f32(agent_state[..., :4])
    asz = None if N == 0 else _lib.as_f32(agent_size)
    aty = None if (N == 0 or agent_type is None) else _lib.as_i32(agent_type)
    per_cam = 0
    pr = None
    if N > 0 and present is not None:
        pr = _lib.as_u8(present)
        per_cam = 1 if pr.dim() == 3 else 0
        if per_cam and tuple(pr.shape) != (B, Nc, N) or (not per_cam and tuple(pr.shape) != (B, N)):
            raise _lib.TdsError("raster: present mask must be [B,N] or [B,Nc,N]")
    tlc = None if L == 0 else _lib.as_f32(tl_corners)
    tls = None if L == 0 else _lib.as_i32(tl_state)
    rc = None if R == 0 else _lib.as_f32(rect_corners)
    rcl = None if R == 0 else _lib.as_i32(rect_class)
    if image_format not in (_lib.IMAGE_F32, _lib.IMAGE_U8, _lib.IMAGE_RANK):
        raise _lib.TdsError(f"raster: unknown image format {image_format}")
    oshape = (B, Nc, res, res) if image_format == _lib.IMAGE_RANK else (B, Nc, 3, res, res)
    odtype = torch.float32 if image_format == _lib.IMAGE_F32 else torch.uint8
    if out is None:
        out = torch.empty(oshape, dtype=odtype, device=dev)
    elif tuple(out.shape) != oshape or out.dtype != odtype or not out.is_contiguous():
        raise _lib.TdsError(f"raster: `out` must be a contiguous {odtype} {list(oshape)} tensor")
    need = lib.tds_raster_workspace_bytes(B, N, L, R)
    if workspace is None or workspace.numel() < need:
        workspace = torch.empty(need, dtype=torch.uint8, device=dev)
    Tc, ctr, ccl = 0, None, None
    if cam_tris is not None and cam_tris.shape[2] > 0:
        Tc = cam_tris.shape[2]
        if tuple(cam_tris.shape) != (B, Nc, Tc, 3, 2) or cam_tri_class is None or tuple(cam_tri_class.shape) != (B, Nc, Tc):
            raise _lib.TdsError("raster: cam_tris must be [B,Nc,Tc,3,2] and cam_tri_class [B,Nc,Tc]")
        ctr, ccl = _lib.as_f32(cam_tris), _lib.as_i32(cam_tri_class)
    acl = None
    if agent_class is not None and N > 0:
        if tuple(agent_class.shape) != (B, Nc, N) or agent_class.dtype != torch.uint8:
            raise _lib.TdsError("raster: agent_class must be uint8 [B,Nc,N]")
        acl = agent_class.contiguous()
    handles, n_maps = mapset.handles(dev)
    env_map = mapset.env_map_on(dev)
    _lib.check(lib.tds_raster_birdview_fmt(handles, n_maps, _lib.ptr(env_map), B, Nc, N, _lib.ptr(cxy), _lib.ptr(csc),
                                           _lib.ptr(ast), _lib.ptr(asz), _lib.ptr(aty), _lib.ptr(pr), per_cam,
                                           _lib.ptr(tlc), _lib.ptr(tls), L, _lib.ptr(rc), _lib.ptr(rcl), R,
                                           _lib.ptr(ctr), _lib.ptr(ccl), Tc, ctypes.byref(palette), float(2.0 / fov), int(res),
                                           _lib.ptr(acl), int(image_format), _lib.ptr(out), _lib.ptr(workspace),
                                           _lib.stream_ptr(dev)))
    return out


def raster_rank_table(palette: "_lib.Palette"):
    """(rgb uint8 [K+1,3], class ids int32 [K+1]) of the draw ranks an IMAGE_RANK image holds: row 0 is the
    background, row k the k-th class in draw order.  rgb[rank_image.long()] is the IMAGE_U8 picture (channels last)."""
    lib = _lib.load()
    rgb = (ctypes.c_uint8 * (3 * (_lib.MAX_CLASSES + 1)))()
    cls = (ctypes.c_int32 * (_lib.MAX_CLASSES + 1))()
    n = lib.tds_raster_rank_table(ctypes.byref(palette), rgb, cls)
    return (torch.tensor(list(rgb), dtype=torch.uint8).reshape(-1, 3)[:n].clone(),
            torch.tensor(list(cls), dtype=torch.int32)[:n].clone())
