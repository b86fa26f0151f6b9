"""The launchers of the range-scan kernels (ops._range_scan_fwd / _range_scan_bwd) check `absolute`, `n_agents`,
`n_rays`, `max_range`, the map set's env_map, kind, idx and the upstream gradient before anything touches the library or
a map handle.  A bad input raises TdsError on the autograd path and on the backward launcher.  CPU tensors suffice: the
checks come before `_lib.load()`, the map handles (which need a CUDA device) and `_lib.ptr()` (which rejects CPU
tensors)."""
import math

import pytest
import torch

import torchdrivesim_b200 as tds
from tests import util
from torchdrivesim_b200 import _lib, ops

Z = torch.zeros
TOWN = tds.MapSet([tds.StaticMap.from_npz(util.map_path("carla_Town02"))])
TWO = tds.MapSet(TOWN.maps * 2, torch.tensor([0, 1, 1]))
LOADED = "the library was loaded before the inputs were checked"


@pytest.fixture(autouse=True)
def no_library(monkeypatch):
    def load(*args, **kwargs):
        raise AssertionError(LOADED)
    monkeypatch.setattr(_lib, "load", load)


def _i64(*shape):
    return torch.full(shape, -1, dtype=torch.int64)


def _forward(absolute, n_rays, n_agents=None, max_range=50.0, mapset=None):
    return lambda: ops.range_scan(absolute.requires_grad_(), n_rays, n_agents, max_range, mapset)


def _backward(absolute, n_rays, kind, idx, grad, n_agents=None, mapset=None):
    return lambda: ops._range_scan_bwd(absolute, n_rays, n_agents, mapset, kind, idx, grad)


ABS = r"absolute must be \[B,N,6\]"
AGENTS = r"n_agents must be in \[0, N\]"
RAYS = r"n_rays must be an integer in \[1, 256\]"
RANGE = r"max_range must be finite and > 0"
ENV = r"env_map must be \[B\]"
KIND = r"kind must be int64 \[B,A,R\]"
IDX = r"idx must be int64 \[B,A,R\]"
GRAD = r"the gradient must be \[B,A,R\]"
CASES = [
    ("absolute-dims", _forward(Z(3, 6), 4), ABS),
    ("absolute-per-origin", _forward(Z(2, 3, 3, 6), 4), ABS),
    ("absolute-columns", _forward(Z(2, 3, 4), 4), ABS),
    ("absolute-columns-backward", _backward(Z(2, 3, 5), 4, _i64(2, 3, 4), _i64(2, 3, 4), Z(2, 3, 4)), ABS),
    ("n-agents-above-n", _forward(Z(2, 3, 6), 4, n_agents=4), AGENTS),
    ("n-agents-negative", _forward(Z(2, 3, 6), 4, n_agents=-1), AGENTS),
    ("n-agents-backward", _backward(Z(2, 3, 6), 4, _i64(2, 4, 4), _i64(2, 4, 4), Z(2, 4, 4), n_agents=4), AGENTS),
    ("rays-zero", _forward(Z(2, 3, 6), 0), RAYS),
    ("rays-negative", _forward(Z(2, 3, 6), -2), RAYS),
    ("rays-above-256", _forward(Z(2, 3, 6), 257), RAYS),
    ("rays-not-integer", _forward(Z(2, 3, 6), 4.0), RAYS),
    ("rays-zero-backward", _backward(Z(2, 3, 6), 0, _i64(2, 3, 0), _i64(2, 3, 0), Z(2, 3, 0)), RAYS),
    ("rays-above-256-backward", _backward(Z(2, 3, 6), 257, _i64(2, 3, 257), _i64(2, 3, 257), Z(2, 3, 257)), RAYS),
    ("range-zero", _forward(Z(2, 3, 6), 4, max_range=0.0), RANGE),
    ("range-negative", _forward(Z(2, 3, 6), 4, max_range=-5.0), RANGE),
    ("range-nan", _forward(Z(2, 3, 6), 4, max_range=math.nan), RANGE),
    ("range-inf", _forward(Z(2, 3, 6), 4, max_range=math.inf), RANGE),
    ("range-float32-overflow", _forward(Z(2, 3, 6), 4, max_range=1e39), RANGE),
    ("range-float32-underflow", _forward(Z(2, 3, 6), 4, max_range=1e-50), RANGE),
    ("env-map-batch", _forward(Z(2, 3, 6), 4, mapset=TWO), ENV),
    ("env-map-batch-backward", _backward(Z(2, 3, 6), 4, _i64(2, 3, 4), _i64(2, 3, 4), Z(2, 3, 4), mapset=TWO), ENV),
    ("kind-rays", _backward(Z(2, 3, 6), 4, _i64(2, 3, 5), _i64(2, 3, 4), Z(2, 3, 4)), KIND),
    ("kind-rows", _backward(Z(2, 3, 6), 4, _i64(2, 2, 4), _i64(2, 3, 4), Z(2, 3, 4)), KIND),
    ("kind-int32", _backward(Z(2, 3, 6), 4, _i64(2, 3, 4).int(), _i64(2, 3, 4), Z(2, 3, 4)), KIND),
    ("idx-rays", _backward(Z(2, 3, 6), 4, _i64(2, 3, 4), _i64(2, 3, 3), Z(2, 3, 4)), IDX),
    ("idx-batch", _backward(Z(2, 3, 6), 4, _i64(2, 3, 4), _i64(1, 3, 4), Z(2, 3, 4)), IDX),
    ("idx-int32", _backward(Z(2, 3, 6), 4, _i64(2, 3, 4), _i64(2, 3, 4).int(), Z(2, 3, 4)), IDX),
    ("grad-rays", _backward(Z(2, 3, 6), 4, _i64(2, 3, 4), _i64(2, 3, 4), Z(2, 3, 5)), GRAD),
    ("grad-rows", _backward(Z(2, 3, 6), 4, _i64(2, 3, 4), _i64(2, 3, 4), Z(2, 2, 4)), GRAD),
    ("grad-extra-dim", _backward(Z(2, 3, 6), 4, _i64(2, 3, 4), _i64(2, 3, 4), Z(2, 3, 4, 1)), GRAD),
]


@pytest.mark.parametrize("call,match", [pytest.param(call, match, id=name) for name, call, match in CASES])
def test_bad_inputs_raise_before_the_library_is_touched(call, match):
    with pytest.raises(_lib.TdsError, match=match):
        call()


def test_well_formed_inputs_reach_the_library():
    """The checks above do not reject a valid call: with a map it gets as far as the map handles, which need a CUDA
    device; without one as far as loading the library."""
    for call in (_forward(Z(2, 3, 6), 256, 2, 5.0, TOWN), _forward(Z(3, 5, 6), 1, mapset=TWO),
                 _backward(Z(2, 3, 6), 4, _i64(2, 3, 4), _i64(2, 3, 4), Z(2, 3, 4), mapset=TOWN)):
        with pytest.raises(_lib.TdsError, match="StaticMap needs a CUDA device"):
            call()
    for call in (_forward(Z(2, 3, 6), 64), _forward(Z(2, 3, 6), 1, 0, 1e-3),
                 _backward(Z(2, 3, 6), 4, _i64(2, 1, 4), _i64(2, 1, 4), Z(2, 1, 4), n_agents=1)):
        with pytest.raises(AssertionError, match=LOADED):
            call()
