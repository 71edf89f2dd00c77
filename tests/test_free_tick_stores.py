"""The force-free FAST tick stores a velocity plane only where its bits changed (SIG_FREE in body_kernels.cu).

A velocity the tick changed must never be dropped.  Reference: an identical executor with a trajectory sample on every
tick — the ring stores every computed value unconditionally — whose last sample must equal the downloaded WorldVel bit
for bit, for degenerate bodies in every position the body-pair kernel treats apart (first pairs, last pairs, the odd
tail, a degenerate partner of a healthy body) and for the one-body-per-thread kernel of small batches.
"""

import numpy as np
import pytest

import elodin_b200 as el
from elodin_b200.executor import WORLD_POS, WORLD_VEL
from tests.util import random_world

pytestmark = pytest.mark.gpu

PAIR_WAVE = 2 * 128 * 3 * 148  # the smallest batch the body-pair kernel takes


@pytest.fixture(autouse=True)
def _need_gpu():
    if el.device_count() < 1:
        pytest.skip("needs a CUDA device")


def _degenerate(pos, vel, ine, b, kind):
    if kind == "zero_mass":
        ine[b, 0, 6] = 0.0
    elif kind == "inf_mass":
        ine[b, 0, 6] = np.inf
    elif kind == "nan_mass":
        ine[b, 0, 6] = np.nan
    elif kind == "denormal_mass":
        ine[b, 0, 6] = 5e-324
    elif kind == "negative_mass":
        ine[b, 0, 6] = -3.0
    elif kind == "zero_ixx":
        ine[b, 0, 0] = 0.0
    elif kind == "neg_zero_vel":
        vel[b, 0, [0, 2, 4]] = -0.0
    elif kind == "nan_vel":
        vel[b, 0, 4] = np.nan
    else:
        raise KeyError(kind)


KINDS = ["zero_mass", "inf_mass", "nan_mass", "denormal_mass", "negative_mass", "zero_ixx", "neg_zero_vel", "nan_vel"]


def _world(M, tail_kind):
    pos, vel, ine = random_world(31, M, 1)
    K = len(KINDS)
    half, quarter = (M // 2) & ~1, (M // 4) & ~1  # pairs are (2t, 2t + 1)
    placed = {}
    for i, kind in enumerate(KINDS):
        for b in (i,                      # first pairs: both bodies of a pair degenerate
                  M - 1 - K + i,          # last pairs before the tail
                  half + 2 * i + 1,       # second body of a pair whose first is healthy
                  quarter + 2 * i):       # first body of a pair whose second is healthy
            _degenerate(pos, vel, ine, b, kind)
            placed.setdefault(kind, []).append(b)
    _degenerate(pos, vel, ine, M - 1, tail_kind)  # the odd tail of the pair kernel
    placed.setdefault(tail_kind, []).append(M - 1)
    healthy = half + 2 * K + 4
    return pos, vel, ine, placed, healthy


def _u64(a):
    return np.ascontiguousarray(a).view(np.uint64)


@pytest.mark.parametrize("M,tail_kind", [(PAIR_WAVE + 3, "zero_mass"), (PAIR_WAVE + 3, "neg_zero_vel"),
                                         (PAIR_WAVE + 3, "nan_vel"), (1001, "nan_mass")])
def test_force_free_tick_never_drops_a_changed_velocity(M, tail_kind):
    pos, vel, ine, placed, healthy = _world(M, tail_kind)
    for b in placed["zero_ixx"] + [healthy]:
        assert np.all(vel[b] != 0.0) and np.isfinite(vel[b]).all()

    def run(traj):
        kw = dict(trajectory_every=1, trajectory_capacity=4) if traj else {}
        with el.B200Exec(1, M, 0.01, None, [], "rk4", "fast", max_fused_ticks=1, **kw) as ex:
            ex.set_state(pos, vel, ine)
            states = []
            for n in (1, 3):  # one launch per tick: consecutive launches walk the planes in opposite directions
                ex.step(n, sync=True)
                states.append((ex.download(WORLD_POS), ex.download(WORLD_VEL)))
            return states, (ex.trajectory() if traj else None)

    got, _ = run(False)
    ref, ring = run(True)
    assert ring.shape == (4, M, 1, 13)
    for (gp, gv), (rp, rv), s in zip(got, ref, (0, 3)):
        assert np.array_equal(_u64(gv), _u64(ring[s][..., 7:13])), s
        assert np.array_equal(_u64(gp), _u64(rp)), s
        assert np.array_equal(_u64(rv), _u64(ring[s][..., 7:13])), s
        assert np.array_equal(_u64(gp), _u64(ring[s][..., :7])), s

    v = got[-1][1]
    # the degenerate bodies really changed: a zero mass turns the linear velocity into NaN, -0.0 becomes +0.0
    for b in placed["zero_mass"]:
        assert np.isnan(v[b, 0, 3:]).all(), b
    for b in placed["neg_zero_vel"]:
        assert not np.signbit(v[b, 0, [0, 2, 4]]).any() and np.signbit(vel[b, 0, [0, 2, 4]]).all(), b
    for b in placed["nan_vel"]:
        assert np.isnan(v[b, 0, 4]), b
    # and a healthy force-free body keeps its velocity bit for bit (nothing was stored into it)
    assert np.array_equal(_u64(v[healthy]), _u64(vel[healthy]))
    assert np.array_equal(_u64(v[placed["zero_ixx"]]), _u64(vel[placed["zero_ixx"]]))
