"""The launchers of the time-to-collision kernels (ops._time_to_collision_fwd / _time_to_collision_bwd) check the shapes
of state, size and present, `n_agents`, the horizon, the index and the upstream gradient before anything touches the
library.  A bad input raises TdsError on every path that reaches a kernel - the autograd Function, the
torch.ops.tds_b200.time_to_collision custom operator and its backward operator.  CPU tensors suffice: the check comes
before `_lib.load()` and `_lib.ptr()` (which rejects CPU tensors)."""
import math

import pytest
import torch

import torchdrivesim_b200  # noqa: F401  (registers torch.ops.tds_b200)
from torchdrivesim_b200 import _lib, ops

OPS = torch.ops.tds_b200
Z = torch.zeros


@pytest.fixture(autouse=True)
def no_library(monkeypatch):
    def load(*args, **kwargs):
        raise AssertionError("the library was loaded before the inputs were checked")
    monkeypatch.setattr(_lib, "load", load)


def _idx(*shape):
    return torch.full(shape, -1, dtype=torch.int64)


def _present(*shape):
    return torch.ones(shape, dtype=torch.bool)


def _ttc(state, size, present, horizon=5.0, n_agents=None, paths=("autograd", "op", "op_backward")):
    """The forward paths (autograd and operator) and the backward operator, with an index and gradient of the shape
    the arguments would give."""
    B = state.shape[0] if state.dim() > 0 else 0
    A = n_agents if isinstance(n_agents, int) and n_agents >= 0 else (state.shape[1] if state.dim() > 1 else 0)
    calls = {"autograd": lambda: ops.time_to_collision(state.requires_grad_(), size, present, horizon, n_agents),
             "op": lambda: OPS.time_to_collision(state, size, present, horizon, n_agents),
             "op_backward": lambda: OPS.time_to_collision_backward(Z(B, A), state, size, present, _idx(B, A), horizon,
                                                                   n_agents)}
    return {p: calls[p] for p in paths}


def _backward(idx, grad, n_agents=2):
    state, size, present = Z(2, 3, 4), Z(2, 3, 2), _present(2, 3)
    return {"op_backward": lambda: OPS.time_to_collision_backward(grad, state, size, present, idx, 3.0, n_agents),
            "launcher": lambda: ops._time_to_collision_bwd(state, size, present, n_agents, 3.0, idx, grad)}


STATE = r"state must be \[B,N,4\]"
SIZE = r"size must be \[B,N,2\]"
PRESENT = r"present must be \[B,N\]"
N_AGENTS = r"n_agents must be an integer in \[0, N\]"
HORIZON = r"horizon must be finite and > 0"
IDX = r"idx must be int64 \[B,A\]"
GRAD = r"the gradient must be \[B,A\]"
CASES = [
    ("state-dims", _ttc(Z(3, 4), Z(3, 2), _present(3)), STATE),
    ("state-four-dims", _ttc(Z(2, 3, 3, 4), Z(2, 3, 2), _present(2, 3)), STATE),
    ("state-columns", _ttc(Z(2, 3, 5), Z(2, 3, 2), _present(2, 3)), STATE),
    ("size-columns", _ttc(Z(2, 3, 4), Z(2, 3, 3), _present(2, 3)), SIZE),
    ("size-agents", _ttc(Z(2, 3, 4), Z(2, 4, 2), _present(2, 3)), SIZE),
    ("size-batch", _ttc(Z(2, 3, 4), Z(1, 3, 2), _present(2, 3)), SIZE),
    ("present-agents", _ttc(Z(2, 3, 4), Z(2, 3, 2), _present(2, 4)), PRESENT),
    ("present-batch", _ttc(Z(2, 3, 4), Z(2, 3, 2), _present(3, 3)), PRESENT),
    ("present-extra-dim", _ttc(Z(2, 3, 4), Z(2, 3, 2), _present(2, 3, 1)), PRESENT),
    ("n-agents-above-n", _ttc(Z(2, 3, 4), Z(2, 3, 2), _present(2, 3), 5.0, 4), N_AGENTS),
    ("n-agents-negative", _ttc(Z(2, 3, 4), Z(2, 3, 2), _present(2, 3), 5.0, -1), N_AGENTS),
    ("n-agents-not-integer", _ttc(Z(2, 3, 4), Z(2, 3, 2), _present(2, 3), 5.0, 1.5, ("autograd",)), N_AGENTS),
    ("horizon-zero", _ttc(Z(2, 3, 4), Z(2, 3, 2), _present(2, 3), 0.0), HORIZON),
    ("horizon-negative", _ttc(Z(2, 3, 4), Z(2, 3, 2), _present(2, 3), -1.0), HORIZON),
    ("horizon-nan", _ttc(Z(2, 3, 4), Z(2, 3, 2), _present(2, 3), math.nan), HORIZON),
    ("horizon-inf", _ttc(Z(2, 3, 4), Z(2, 3, 2), _present(2, 3), math.inf), HORIZON),
    ("horizon-float32-overflow", _ttc(Z(2, 3, 4), Z(2, 3, 2), _present(2, 3), 1e39), HORIZON),
    ("horizon-float32-underflow", _ttc(Z(2, 3, 4), Z(2, 3, 2), _present(2, 3), 1e-50), HORIZON),
    ("idx-rows", _backward(_idx(2, 3), Z(2, 2)), IDX),
    ("idx-batch", _backward(_idx(1, 2), Z(2, 2)), IDX),
    ("idx-extra-dim", _backward(_idx(2, 2, 1), Z(2, 2)), IDX),
    ("idx-int32", _backward(_idx(2, 2).int(), Z(2, 2)), IDX),
    ("idx-float", _backward(Z(2, 2), Z(2, 2)), IDX),
    ("grad-rows", _backward(_idx(2, 2), Z(2, 3)), GRAD),
    ("grad-batch", _backward(_idx(2, 2), Z(1, 2)), GRAD),
    ("grad-extra-dim", _backward(_idx(2, 2), Z(2, 2, 1)), GRAD),
]


@pytest.mark.parametrize("call,match", [pytest.param(call, match, id=f"{name}-{path}")
                                        for name, paths, match in CASES for path, call in paths.items()])
def test_bad_inputs_raise_before_the_library_is_touched(call, match):
    with pytest.raises(_lib.TdsError, match=match):
        call()


def test_well_formed_inputs_reach_the_library():
    """The checks above do not reject a valid call: it gets as far as the library (here: the failing loader)."""
    state, size, present = Z(2, 3, 4), Z(2, 3, 2), _present(2, 3)
    for call in (lambda: ops.time_to_collision(state, size, present),
                 lambda: ops.time_to_collision(state, size, present.to(torch.uint8), 0.5, 0),
                 lambda: OPS.time_to_collision(state, size, present, 8.0, 3),
                 lambda: OPS.time_to_collision_backward(Z(2, 2), state, size, present, _idx(2, 2), 3.0, 2),
                 lambda: OPS.time_to_collision_backward(Z(2, 3), state, size, present, _idx(2, 3), 3.0, None)):
        with pytest.raises(AssertionError, match="the library was loaded"):
            call()
