"""Time to collision on the GPU (ops.time_to_collision, tds_time_to_collision and its backward).

The forward is compared bit for bit (ttc bits and idx) with an eager torch float32 statement of its definition over
all pairs, one op per operation (each rounds on its own, as the definition asks); the headings' sin / cos are those of
ops.egocentric_cameras, the library's double-precision sincos rounded to float32.  Independently of the SAT formula,
the winners are checked against the float64 box clipping of oracle/iou.py: the boxes overlap just after the reported
time and nothing overlaps the origin just before it.  The backward is compared with float64 autograd of
t = -(d0 + sgn(s) R) / s on the winning axis."""
import math

import numpy as np
import pytest
import torch

import torchdrivesim_b200 as tds
from oracle import iou as OI
from tests import util
from tests.test_gpu_observation_grads import check
from torchdrivesim_b200 import ops

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
EMPTY = (1 << 63) - 1


def _bits(t):
    return t.contiguous().view(torch.int32)


# ------------------------------------------------------------------------------------------------ the definition
def sincos(state):
    """(sin psi, cos psi) [B,N] of the library (double precision, rounded to float32)."""
    sc = ops.egocentric_cameras(state.contiguous())[1]
    return sc[..., 0], sc[..., 1]


def ttc_ref(state, size, present, A, horizon):
    """(ttc [B,A], idx [B,A], axis [B,A], s on that axis [B,A]) of the definition, float32, every op on its own."""
    B, N = state.shape[:2]
    H = float(np.float32(horizon))
    sn, cs = sincos(state)
    x, y, v = state[..., 0], state[..., 1], state[..., 3]
    vx, vy = v * cs, v * sn
    hl, hw = 0.5 * size[..., 0], 0.5 * size[..., 1]

    def I(t):
        return t[:, :A, None]

    def J(t):
        return t[:, None, :]

    inf = torch.tensor(math.inf, device=DEV)
    entries, exits, svs = [], [], []
    never = torch.zeros(B, A, N, dtype=torch.bool, device=DEV)
    for k in range(4):
        own, oth = (I, J) if k < 2 else (J, I)
        nx = -own(sn) if k & 1 else own(cs)
        ny = own(cs) if k & 1 else own(sn)
        p = nx * oth(cs) + ny * oth(sn)
        q = nx * (-oth(sn)) + ny * oth(cs)
        h_own = own(hw) if k & 1 else own(hl)
        h_oth = p.abs() * oth(hl) + q.abs() * oth(hw)
        R = h_own + h_oth if k < 2 else h_oth + h_own
        d0 = nx * (J(x) - I(x)) + ny * (J(y) - I(y))
        sv = nx * (J(vx) - I(vx)) + ny * (J(vy) - I(vy))
        ta = (-R - d0) / sv
        tb = (R - d0) / sv
        nz = sv != 0
        entries.append(torch.where(nz, torch.minimum(ta, tb), -inf))
        exits.append(torch.where(nz, torch.maximum(ta, tb), inf))
        svs.append(sv.expand(B, A, N))
        never |= ~nz & ~(d0.abs() <= R)
    en = torch.stack(entries)
    t_in, t_out = en.amax(0), torch.stack(exits).amin(0)
    zero = torch.zeros((), device=DEV)
    touch = torch.maximum(t_in, zero) <= torch.minimum(t_out, torch.tensor(H, device=DEV))
    j = torch.arange(N, device=DEV)
    valid = (j[None, None, :] != torch.arange(A, device=DEV)[None, :, None]) & I(present) & J(present)
    touch = touch & ~never & valid
    t = torch.where(t_in > 0, t_in, zero)
    word = torch.where(touch, (_bits(t).long() << 32) | j, EMPTY)
    best, arg = word.min(-1)
    none = best == EMPTY
    ttc = torch.where(none, math.inf, (best >> 32).int().view(torch.float32))
    idx = torch.where(none, -1, best & 0xFFFFFFFF)
    # the first axis whose entry is T_in, and its s, for the winning pair
    win_en = en.gather(3, arg[None, :, :, None].expand(4, B, A, 1))[..., 0]
    win_tin = t_in.gather(2, arg[..., None])[..., 0]
    axis = (win_en == win_tin[None]).int().argmax(0)
    sv = torch.stack(svs).gather(3, arg[None, :, :, None].expand(4, B, A, 1))[..., 0].gather(0, axis[None])[0]
    return ttc, idx, axis, sv


def _assert_same(got, ref):
    ttc, idx = got
    assert ttc.dtype == torch.float32 and idx.dtype == torch.int64
    assert torch.equal(idx, ref[1])
    assert torch.equal(_bits(ttc), _bits(ref[0]))


def crowd(rng, B, N, box=120.0, vmax=15.0):
    """state [B,N,4], size [B,N,2], present [B,N]: agents uniform in a box-metre square, random headings and speeds,
    vehicle-like sizes, 10 % absent."""
    state = np.concatenate([rng.uniform(0, box, (B, N, 2)), rng.uniform(-np.pi, np.pi, (B, N, 1)),
                            rng.uniform(0, vmax, (B, N, 1))], -1).astype(np.float32)
    size = np.stack([rng.uniform(3.5, 6.0, (B, N)), rng.uniform(1.6, 2.6, (B, N))], -1).astype(np.float32)
    present = rng.uniform(size=(B, N)) > 0.1
    return (torch.tensor(state, device=DEV), torch.tensor(size, device=DEV), torch.tensor(present, device=DEV))


def bench_inputs():
    import bench
    state, size, _, _ = bench.synth_inputs(1024, 64, 0, 1)
    return (torch.tensor(state, device=DEV), torch.tensor(size, device=DEV),
            torch.ones(1024, 64, dtype=torch.bool, device=DEV))


# ------------------------------------------------------------------------------------------------ forward
@pytest.mark.parametrize("H", [0.5, 3.0, 8.0])
def test_random_crowds_are_the_definition(H):
    rng = np.random.default_rng(int(H * 10))
    state, size, present = crowd(rng, 64, 512)
    got = ops.time_to_collision(state, size, present, H)
    ref = ttc_ref(state, size, present, 512, H)
    _assert_same(got, ref)
    assert (got[1] >= 0).any() and (got[1] == -1).any() and (got[0] > 0).any()


@pytest.mark.parametrize("H", [0.5, 3.0, 8.0])
def test_config2_inputs_are_the_definition(H):
    state, size, present = bench_inputs()
    _assert_same(ops.time_to_collision(state, size, present, H), ttc_ref(state, size, present, 64, H))


def test_npcs_absent_zero_size_and_nan_rows():
    rng = np.random.default_rng(3)
    state, size, present = crowd(rng, 4, 96, box=40.0)
    state[0, 1, 0] = math.nan
    state[1, 2, 2] = math.nan
    state[2, 3, 3] = math.nan
    state[3, 4, 1] = math.inf
    state[0, 70, 0] = math.nan                                     # an NPC
    size[0, 5] = 0.0
    size[1, 6, 0] = math.nan
    size[2, 80] = 0.0
    present[:, 7] = False
    got = ops.time_to_collision(state, size, present, 3.0, 60)
    _assert_same(got, ttc_ref(state, size, present, 60, 3.0))
    assert (got[1][:, 7] == -1).all() and torch.isinf(got[0][:, 7]).all()
    assert (got[1] >= 60).any()                                    # NPCs are candidates
    assert not ((got[1] == 7).any())


def test_no_origins_and_one_agent():
    rng = np.random.default_rng(4)
    state, size, present = crowd(rng, 3, 5)
    ttc, idx = ops.time_to_collision(state, size, present, 3.0, 0)
    assert ttc.shape == idx.shape == (3, 0)
    ttc, idx = ops.time_to_collision(state[:, :1], size[:, :1], present[:, :1], 3.0)
    assert torch.isinf(ttc).all() and (idx == -1).all()
    gs, gz = ops._time_to_collision_bwd(state, size, present, 0, 3.0, idx[:, :0], ttc[:, :0])
    assert (gs == 0).all() and (gz == 0).all()


@pytest.mark.parametrize("H", [0.5, 3.0, 8.0])
def test_standing_still(H):
    rng = np.random.default_rng(5)
    state, size, present = crowd(rng, 8, 64, box=30.0)
    state[..., 3] = 0.0
    got = ops.time_to_collision(state, size, present, H)
    _assert_same(got, ttc_ref(state, size, present, 64, H))
    hit = got[1] >= 0
    assert hit.any() and (got[0][hit] == 0).all()                  # only pairs that overlap already


def tie_scene():
    """0 at the origin heading +x at 10 m/s; 1 and 2 identical, 20 m ahead and facing it (equal times: 1 wins);
    3 heads +x alongside 4, which overlaps it (time 0 both ways); 5 and 6 both overlap 7 (7 picks 5), 5 and 6 overlap
    too; 8 stands still 30 m ahead of 9, which drives at it; 10 is 8's copy, absent."""
    rows = [[0, 0, 0, 10], [20, 0, math.pi, 10], [20, 0, math.pi, 10], [0, 50, 0, 5], [2, 50.5, 0, 7],
            [100, 0, 1, 3], [101, 0, 2, 3], [100.5, 0.5, 0, 0], [200, 0, 0, 0], [170, 0, 0, 10], [200, 0, 0, 0]]
    state = torch.tensor([rows], dtype=torch.float32, device=DEV)
    size = torch.tensor([[[4, 2]] * len(rows)], dtype=torch.float32, device=DEV)
    present = torch.ones(1, len(rows), dtype=torch.bool, device=DEV)
    present[0, 10] = False
    return state, size, present


@pytest.mark.parametrize("H", [0.5, 3.0, 8.0])
def test_overlaps_and_ties(H):
    state, size, present = tie_scene()
    ttc, idx = ops.time_to_collision(state, size, present, H)
    _assert_same((ttc, idx), ttc_ref(state, size, present, state.shape[1], H))
    assert float(ttc[0, 3]) == 0.0 and int(idx[0, 3]) == 4 and float(ttc[0, 4]) == 0.0 and int(idx[0, 4]) == 3
    assert float(ttc[0, 7]) == 0.0 and int(idx[0, 7]) == 5 and int(idx[0, 5]) == 6 and int(idx[0, 6]) == 5
    assert (_bits(ttc) != _bits(torch.tensor(-0.0, device=DEV))).all()
    if H >= 3.0:
        assert int(idx[0, 0]) == 1 and abs(float(ttc[0, 0]) - 0.8) < 1e-6 and float(ttc[0, 1]) == float(ttc[0, 2])
        assert int(idx[0, 9]) == 8 and abs(float(ttc[0, 9]) - 2.6) < 1e-5 and int(idx[0, 8]) == 9
    else:
        assert int(idx[0, 0]) == -1 and int(idx[0, 9]) == -1


def test_more_than_one_tile_of_columns():
    rng = np.random.default_rng(6)
    state, size, present = crowd(rng, 2, 2100, box=250.0)
    for A in (2100, 300):
        got = ops.time_to_collision(state, size, present, 3.0, A)
        ref = ttc_ref(state, size, present, A, 3.0)
        _assert_same(got, ref)
        assert (got[1] >= 1024).any() and (got[1][:, :64] >= 0).any()


# ------------------------------------------------------------------------------------------------ known answers
def _pair(a, b, H):
    state = torch.tensor([[a, b]], dtype=torch.float32, device=DEV)
    size = torch.tensor([[[4, 2], [4, 2]]], dtype=torch.float32, device=DEV)
    present = torch.ones(1, 2, dtype=torch.bool, device=DEV)
    ttc, idx = ops.time_to_collision(state, size, present, H)
    _assert_same((ttc, idx), ttc_ref(state, size, present, 2, H))
    return ttc[0].tolist(), idx[0].tolist()


def test_known_answers():
    # head on, 20 m apart at 10 m/s each: the fronts close 16 m at 20 m/s
    ttc, idx = _pair([0, 0, 0, 10], [20, 0, math.pi, 10], 5.0)
    assert idx == [1, 0] and all(abs(t - 0.8) < 1e-6 for t in ttc)
    ttc, idx = _pair([0, 0, 0, 10], [20, 0, math.pi, 10], 0.5)
    assert idx == [-1, -1] and all(math.isinf(t) for t in ttc)
    # same lane, same speed: never
    ttc, idx = _pair([0, 0, 0, 10], [10, 0, 0, 10], 8.0)
    assert idx == [-1, -1] and all(math.isinf(t) for t in ttc)
    # perpendicular crossing: j 20 m ahead and 20 m to the right, driving left across i's path.  Relative position
    # (20, -20), relative velocity (-10, 10); on x the gap closes from 20 to 2 + 1 = 3 m at 1.7 s, on y from 20 to
    # 1 + 2 = 3 m at 1.7 s too, and both stay closed until 2.3 s
    ttc, idx = _pair([0, 0, 0, 10], [20, -20, math.pi / 2, 10], 5.0)
    assert idx == [1, 0] and all(abs(t - 1.7) < 1e-5 for t in ttc)
    # ... 5 m further down: x closes at 1.7 s, y only at 2.2 s
    ttc, idx = _pair([0, 0, 0, 10], [20, -25, math.pi / 2, 10], 5.0)
    assert idx == [1, 0] and all(abs(t - 2.2) < 1e-5 for t in ttc)


# ------------------------------------------------------------------------------------------------ geometry
def _corners(state, size, t):
    """[P,4,2] float64 corners of the boxes at time t [P] under constant velocity (oracle/iou.py's corner order)."""
    st = state.astype(np.float64)
    x = st[:, 0] + t * st[:, 3] * np.cos(st[:, 2])
    y = st[:, 1] + t * st[:, 3] * np.sin(st[:, 2])
    return OI.corners(np.stack([x, y, size[:, 0].astype(np.float64), size[:, 1].astype(np.float64), st[:, 2]], -1))


# oracle/iou.py counts a vertex within 1e-6 of the other box's normalised extent as inside, so two boxes that do not
# overlap can show a sliver of that width; an overlap that the reported TTC missed is far larger
NO_OVERLAP = 1e-6


@pytest.mark.parametrize("H", [3.0, 8.0])
def test_winners_touch_and_nothing_comes_first(H):
    rng = np.random.default_rng(11 + int(H))
    state, size, present = crowd(rng, 8, 128, box=60.0)
    ttc, idx = ops.time_to_collision(state, size, present, H)
    st, sz, pr = state.cpu().numpy(), size.cpu().numpy(), present.cpu().numpy()
    t, j = ttc.cpu().numpy().astype(np.float64), idx.cpu().numpy()
    b, i = np.nonzero(j >= 0)
    assert len(b) > 50
    after = t[b, i] * (1 + 1e-4) + 1e-4
    area = OI.intersection_area(_corners(st[b, i], sz[b, i], after), _corners(st[b, j[b, i]], sz[b, j[b, i]], after))
    assert (area > 0).all()
    # no candidate of an origin overlaps it just before its TTC
    keep = t[b, i] > 1e-3
    b, i = b[keep], i[keep]
    before = t[b, i] * (1 - 1e-4) - 1e-4
    N = st.shape[1]
    bb, ii, jj = np.repeat(b, N), np.repeat(i, N), np.tile(np.arange(N), len(b))
    tt = np.repeat(before, N)
    ok = (jj != ii) & pr[bb, jj]
    bb, ii, jj, tt = bb[ok], ii[ok], jj[ok], tt[ok]
    area = OI.intersection_area(_corners(st[bb, ii], sz[bb, ii], tt), _corners(st[bb, jj], sz[bb, jj], tt))
    assert (area < NO_OVERLAP).all()


def test_no_pair_overlaps_before_its_ttc_on_a_time_grid():
    rng = np.random.default_rng(12)
    H = 3.0
    state, size, present = crowd(rng, 2, 12, box=25.0, vmax=10.0)
    ttc, idx = ops.time_to_collision(state, size, present, H)
    st, sz, pr = state.cpu().numpy(), size.cpu().numpy(), present.cpu().numpy()
    t = ttc.cpu().numpy().astype(np.float64)
    assert (idx >= 0).sum() >= 4
    grid = np.linspace(0.0, H, 301)
    B, N = pr.shape
    bb, ii, jj = np.meshgrid(np.arange(B), np.arange(N), np.arange(N), indexing="ij")
    bb, ii, jj = bb.ravel(), ii.ravel(), jj.ravel()
    ok = (ii != jj) & pr[bb, ii] & pr[bb, jj]
    bb, ii, jj = bb[ok], ii[ok], jj[ok]
    tg = np.repeat(grid, len(bb))
    bb, ii, jj = np.tile(bb, len(grid)), np.tile(ii, len(grid)), np.tile(jj, len(grid))
    early = tg < t[bb, ii] * (1 - 1e-4) - 1e-4
    bb, ii, jj, tg = bb[early], ii[early], jj[early], tg[early]
    area = OI.intersection_area(_corners(st[bb, ii], sz[bb, ii], tg), _corners(st[bb, jj], sz[bb, jj], tg))
    assert (area < NO_OVERLAP).all()


# ------------------------------------------------------------------------------------------------ backward
def grad_ref(state, size, present, A, ttc, idx, axis, g):
    """float64 autograd of t = -(d0 + sgn(s) R) / s on the winning axis -> (d state [B,N,4], d size [B,N,2], S [B,N,6]:
    per element, the magnitudes of the terms entering it times the conditioning of t, for check())."""
    B, N = state.shape[:2]
    xs = state.double().clone().requires_grad_()
    xz = size.double().clone().requires_grad_()
    rows = (ttc > 0) & torch.isfinite(ttc) & (idx >= 0)
    bb, ii = torch.nonzero(rows, as_tuple=True)
    jj, kk = idx[bb, ii], axis[bb, ii].long()
    si, sj = xs[bb, ii], xs[bb, jj]
    zi, zj = xz[bb, ii], xz[bb, jj]
    ci, sni, cj, snj = torch.cos(si[:, 2]), torch.sin(si[:, 2]), torch.cos(sj[:, 2]), torch.sin(sj[:, 2])
    own_i = kk < 2
    oc, os_ = torch.where(own_i, ci, cj), torch.where(own_i, sni, snj)
    tc, ts = torch.where(own_i, cj, ci), torch.where(own_i, snj, sni)
    perp = (kk % 2) == 1
    nx, ny = torch.where(perp, -os_, oc), torch.where(perp, oc, os_)
    p, q = nx * tc + ny * ts, -nx * ts + ny * tc
    own_hl, own_hw = torch.where(own_i, zi[:, 0], zj[:, 0]), torch.where(own_i, zi[:, 1], zj[:, 1])
    oth_hl, oth_hw = torch.where(own_i, zj[:, 0], zi[:, 0]), torch.where(own_i, zj[:, 1], zi[:, 1])
    R = 0.5 * torch.where(perp, own_hw, own_hl) + 0.5 * (p.abs() * oth_hl + q.abs() * oth_hw)
    dx, dy = sj[:, 0] - si[:, 0], sj[:, 1] - si[:, 1]
    dvx, dvy = sj[:, 3] * cj - si[:, 3] * ci, sj[:, 3] * snj - si[:, 3] * sni
    d0 = nx * dx + ny * dy
    s = nx * dvx + ny * dvy
    t = -(d0 + torch.sign(s) * R) / s
    gg = g[bb, ii].double()
    (t * gg).sum().backward()
    with torch.no_grad():
        mag = (1 + dx.abs() + dy.abs() + si[:, 3].abs() + sj[:, 3].abs() + zi.abs().sum(-1) + zj.abs().sum(-1)
               + t.abs() * (dvx.abs() + dvy.abs()))
        K = gg.abs() / s.abs() * (1 + (d0.abs() + R.abs()) / s.abs()) * mag
        S = torch.zeros(B, N, 6, dtype=torch.float64, device=DEV)
        S.index_put_((bb, ii), K[:, None].expand(-1, 6), accumulate=True)
        S.index_put_((bb, jj), K[:, None].expand(-1, 6), accumulate=True)
    return xs.grad, xz.grad, S


@pytest.mark.parametrize("H", [3.0, 8.0])
@pytest.mark.parametrize("shape", [(64, 512), (16, 1100)], ids=["64x512", "16x1100"])
def test_backward_vs_float64_autograd(shape, H):
    B, N = shape
    rng = np.random.default_rng(N + int(H))
    state, size, present = crowd(rng, B, N, box=120.0 if N == 512 else 160.0)
    A = N - 40
    xs, xz = state.clone().requires_grad_(), size.clone().requires_grad_()
    ttc, idx = ops.time_to_collision(xs, xz, present, H, A)
    _, ref_idx, axis, sv = ttc_ref(state, size, present, A, H)
    assert torch.equal(idx, ref_idx)
    g = torch.tensor(rng.standard_normal((B, A)).astype(np.float32), device=DEV)
    g = torch.where(sv.abs() >= 0.1, g, 0.0)                       # well-conditioned pairs only
    gs, gz = torch.autograd.grad(ttc, (xs, xz), g)
    live = (ttc > 0) & torch.isfinite(ttc) & (g != 0)
    assert live.sum() > 100
    ref_s, ref_z, S = grad_ref(state, size, present, A, ttc, idx, axis, g)
    check(torch.cat([gs, gz], -1), torch.cat([ref_s, ref_z], -1), S, terms=A + 1)
    again = ops._time_to_collision_bwd(state, size, present, A, H, idx, g)
    assert torch.equal(_bits(again[0]), _bits(gs)) and torch.equal(_bits(again[1]), _bits(gz))


def test_rows_without_a_positive_time_contribute_nothing():
    rng = np.random.default_rng(13)
    state, size, present = crowd(rng, 8, 256, box=60.0)
    ttc, idx = ops.time_to_collision(state, size, present, 3.0)
    dead = (ttc == 0) | (idx == -1)
    assert (ttc == 0).any() and (idx == -1).any() and (~dead).any()
    g = torch.randn(8, 256, device=DEV)
    g_nan = torch.where(dead, math.nan, g)
    g_inf = torch.where(dead, math.inf, g)
    g_zero = torch.where(dead, 0.0, g)
    ref = ops._time_to_collision_bwd(state, size, present, None, 3.0, idx, g_zero)
    for gg in (g_nan, g_inf):
        got = ops._time_to_collision_bwd(state, size, present, None, 3.0, idx, gg)
        assert torch.isfinite(got[0]).all() and torch.isfinite(got[1]).all()
        assert torch.equal(_bits(got[0]), _bits(ref[0])) and torch.equal(_bits(got[1]), _bits(ref[1]))
    none = ops._time_to_collision_bwd(state, size, present, None, 3.0, torch.full_like(idx, -1), g)
    assert (none[0] == 0).all() and (none[1] == 0).all()


def test_custom_operator():
    rng = np.random.default_rng(14)
    state, size, present = crowd(rng, 3, 24, box=30.0)
    for H, A in ((3.0, 24), (8.0, 17)):
        xs, xz = state.clone().requires_grad_(), size.clone().requires_grad_()
        torch.library.opcheck(torch.ops.tds_b200.time_to_collision.default, (xs, xz, present, H, A))
        ttc, idx = torch.ops.tds_b200.time_to_collision(xs, xz, present, H, A)
        g = torch.where(torch.isfinite(ttc), torch.randn_like(ttc), 0.0)
        got = torch.autograd.grad(ttc, (xs, xz), g)
        ref_ttc, ref_idx = ops.time_to_collision(xs, xz, present, H, A)
        ref = torch.autograd.grad(ref_ttc, (xs, xz), g)
        assert torch.equal(ttc, ref_ttc) and torch.equal(idx, ref_idx)
        assert torch.equal(got[0], ref[0]) and torch.equal(got[1], ref[1])


# ------------------------------------------------------------------------------------------------ Simulator, graphs
def test_simulator_time_to_collision_with_npcs_reaches_the_actions():
    rng = np.random.default_rng(15)
    B, A, npcs = 2, 16, 6
    m = util.load_map_np("carla_Town01")
    state, size, _, present = util.random_scene(m, B, A, rng, spread=6.0, absent_p=0.2)
    log = np.concatenate([state[:, :npcs, None, :2] + rng.normal(0, 6, (B, npcs, 3, 2)), rng.uniform(0, 5, (B, npcs, 3, 2))], -1)
    ctrl = tds.ReplayController(torch.full((B, npcs, 2), 2.0, device=DEV), torch.tensor(log, dtype=torch.float32, device=DEV),
                                torch.tensor(rng.uniform(size=(B, npcs, 3)) > 0.2, device=DEV))
    km = tds.KinematicBicycle(left_handed=True)
    km.set_params(lr=torch.full((B, A), util.VEH[2], device=DEV))
    km.set_state(torch.tensor(state, device=DEV))
    sim = tds.Simulator(tds.StaticMap.from_npz(util.map_path("carla_Town01")), km, torch.tensor(size, device=DEV),
                        torch.tensor(present, device=DEV), tds.TorchDriveConfig(left_handed_coordinates=True),
                        npc_controller=ctrl)
    action = torch.tensor(rng.uniform(-1, 1, (B, A, 2)).astype(np.float32), device=DEV, requires_grad=True)
    sim.step(action)
    ttc, idx = sim.compute_time_to_collision(8.0)
    ref = ops.time_to_collision(sim.get_all_agent_state().detach(), sim.get_all_agent_size()[..., :2].detach(),
                                sim.get_all_agent_present_mask(), 8.0, A)
    assert torch.equal(_bits(ttc), _bits(ref[0])) and torch.equal(idx, ref[1])
    assert ttc.shape == (B, A) and (idx >= 0).any()
    live = (ttc > 0) & torch.isfinite(ttc)
    assert live.any()
    torch.where(live, ttc, 0.0).sum().backward()
    assert action.grad is not None and torch.isfinite(action.grad).all() and (action.grad != 0).any()


def test_cuda_graph_capture_replays_the_eager_result():
    rng = np.random.default_rng(16)
    state, size, present = crowd(rng, 4, 200, box=60.0)
    A = 150
    eager = ops._time_to_collision_fwd(state, size, present, A, 3.0)
    g_in = torch.randn(4, A, device=DEV)
    eager_bwd = ops._time_to_collision_bwd(state, size, present, A, 3.0, eager[1], g_in)
    static = state.clone()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        ops._time_to_collision_fwd(static, size, present, A, 3.0)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = ops._time_to_collision_fwd(static, size, present, A, 3.0)
        gout = ops._time_to_collision_bwd(static, size, present, A, 3.0, out[1], g_in)
    static.copy_(torch.zeros_like(state))
    graph.replay()
    static.copy_(state)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(_bits(out[0]), _bits(eager[0])) and torch.equal(out[1], eager[1])
    assert torch.equal(_bits(gout[0]), _bits(eager_bwd[0])) and torch.equal(_bits(gout[1]), _bits(eager_bwd[1]))
