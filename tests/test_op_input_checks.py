"""The launchers of the differentiable kernels (ops.py) check that their inputs agree in shape before anything touches
the library.  A mismatch raises TdsError on every path that reaches a kernel - the autograd Functions, the `out=` paths
and the torch.ops.tds_b200 custom operators - instead of a launch that reads past the end of the smaller tensor.  CPU
tensors suffice: the check comes before `_lib.load()`, `_lib.ptr()` (which rejects CPU tensors) and the map handles
(which need a CUDA device)."""
import pytest
import torch

import torchdrivesim_b200 as tds
from tests import util
from torchdrivesim_b200 import _lib, ops

OPS = torch.ops.tds_b200
Z = torch.zeros
TOWN = tds.MapSet([tds.StaticMap.from_npz(util.map_path("carla_Town02"))])


@pytest.fixture(autouse=True)
def no_library(monkeypatch):
    def load(*args, **kwargs):
        raise AssertionError("the library was loaded before the input shapes were checked")
    monkeypatch.setattr(_lib, "load", load)


def _kinematic(state, action, lr, model=None):
    return {"autograd": lambda: ops.kinematic_step(state, action, lr, model),
            "out": lambda: ops.kinematic_step(state, action, lr, model, out=torch.empty(state.shape)),
            "op": lambda: OPS.kinematic_step(state, action, lr, model, 0, 0.1, False),
            "op_backward": lambda: OPS.kinematic_step_backward(Z(state.shape), state, action, lr, model, 0, 0.1, False)}


def _pairwise(box1, box2):
    return {"autograd": lambda: ops.collision_pairwise(box1, box2),
            "op": lambda: OPS.collision_pairwise(box1, box2, 0),
            "op_backward": lambda: OPS.collision_pairwise_backward(Z(box1.shape[:-1]), box1, box2, 0)}


def _allpairs(ego, all_box, mask, argmax=None):
    """The forward paths and the backward operator; with `argmax`, the backward operator alone (the autograd paths take
    their argmax from the forward)."""
    backward = lambda: OPS.collision_allpairs_backward(Z(ego.shape[:2]), ego, all_box, mask,  # noqa: E731
                                                       Z(ego.shape[:2], dtype=torch.int32) if argmax is None else argmax, 0, True)
    if argmax is not None:
        return {"op_backward": backward}
    return {"autograd": lambda: ops.collision_allpairs(ego, all_box, mask),
            "out": lambda: ops.collision_allpairs(ego, all_box, mask, out=torch.empty(ego.shape[:2])),
            "op": lambda: OPS.collision_allpairs(ego, all_box, mask, 0, True),
            "op_backward": backward}


def _agent_boxes(state, size):
    return {"autograd": lambda: ops.agent_boxes(state, size),
            "op": lambda: OPS.agent_boxes(state, size)}


def _offroad(state, lenwid, present):
    return {"autograd": lambda: ops.offroad(state, lenwid, TOWN, 0.5, present),
            "out": lambda: ops.offroad(state, lenwid, TOWN, 0.5, present, out=torch.empty(state.shape[:2]))}


MASK = Z(2, 3, dtype=torch.bool)
CASES = [
    ("kinematic-action-rows", _kinematic(Z(4, 4), Z(2, 2), Z(4)), "must agree on the batch shape"),
    ("kinematic-lr-rows", _kinematic(Z(4, 4), Z(4, 2), Z(2)), "must agree on the batch shape"),
    ("kinematic-model-rows", _kinematic(Z(4, 4), Z(4, 2), Z(4), Z(2, dtype=torch.int32)), "must agree on the batch shape"),
    ("pairwise-rows", _pairwise(Z(4, 5), Z(2, 5)), "boxes must have identical shape"),
    ("allpairs-ego-dims", _allpairs(Z(2, 5), Z(2, 3, 5), MASK), r"expected ego_box \[B,A,5\] and all_box \[B,N,5\]"),
    ("allpairs-all-columns", _allpairs(Z(2, 3, 5), Z(2, 3, 4), MASK), r"expected ego_box \[B,A,5\] and all_box \[B,N,5\]"),
    ("allpairs-batch", _allpairs(Z(2, 3, 5), Z(1, 3, 5), MASK), "batch / mask shape mismatch"),
    ("allpairs-mask", _allpairs(Z(2, 3, 5), Z(2, 3, 5), Z(2, 2, dtype=torch.bool)), "batch / mask shape mismatch"),
    ("allpairs-argmax", _allpairs(Z(2, 3, 5), Z(2, 3, 5), MASK, Z(2, 2, dtype=torch.int32)), r"argmax must be \[B,A\]"),
    ("agent-boxes-size-batch", _agent_boxes(Z(2, 3, 4), Z(2, 2, 2)), "expected state .* and size"),
    ("offroad-present", _offroad(Z(2, 3, 4), Z(2, 3, 2), Z(2, 2, dtype=torch.bool)), r"expected present \[B,A\]"),
]


@pytest.mark.parametrize("call,match", [pytest.param(call, match, id=f"{name}-{path}")
                                        for name, paths, match in CASES for path, call in paths.items()])
def test_mismatched_shapes_raise_before_the_library_is_touched(call, match):
    with pytest.raises(_lib.TdsError, match=match):
        call()
