"""GPU: the estimator's filters inside cassie_sim_step_pd(_batch) (pelvis.position / translationalVelocity / externalForce, terrain.height)
against the REAL estimator archive's outputs (tests/golden/archive_runs.npz) and the oracle's restatement."""
import os

import numpy as np
import pytest

from conftest import GOLDEN, PD_DGAIN, PD_PGAIN, PD_TARGET, product

pytestmark = pytest.mark.gpu


def _pd(P):
    pu = P.pd_in_t()
    for side, leg in enumerate((pu.leftLeg, pu.rightLeg)):
        for i in range(5):
            leg.motorPd.pTarget[i] = PD_TARGET[5 * side + i]
            leg.motorPd.pGain[i], leg.motorPd.dGain[i] = PD_PGAIN[i], PD_DGAIN[i]
    return pu


def _filtered(y):
    return np.concatenate([y.pelvis.position[:], y.pelvis.translationalVelocity[:], y.pelvis.externalForce[:], [y.terrain.height]])


def test_filtered_outputs_match_the_estimator(oracle_mod):
    """every call against the oracle's restatement; every 50th call against the real archive's output on the same run (tests/golden/archive_runs.npz)"""
    P, O = product(), oracle_mod
    V = np.load(os.path.join(GOLDEN, 'archive_runs.npz'))
    ticks = list(V['pd_tick'])
    o = O.OracleSim(os.path.join(GOLDEN, 'cassie.omodel'))
    c = P.CassieSim()
    u, pu, y = O.make_pd(pTarget=PD_TARGET, pGain=PD_PGAIN, dGain=PD_DGAIN), _pd(P), P.state_out_t()
    worst = 0.0
    for k in range(700):
        o.step_pd(u, y)
        yc = c.step_pd(pu)
        b = _filtered(yc)
        for a in [_filtered(y)] + ([_filtered(P.state_out_t.from_buffer_copy(V['pd_state_out'][ticks.index(k)].tobytes()))] if k in ticks else []):
            worst = max(worst, (np.abs(a - b) / (1 + np.abs(a))).max())
    # the leg forces feeding the filters agree with the archive only to its single precision: 1e-3 relative is the bar (CPU twin: 1e-4)
    assert worst < 2e-3, worst
    assert abs(b[2]) > 0.3 and abs(b[8] - 31 * 9.806) > 10 and b[9] != 0 and yc.leftFoot.toeForce[2] < -50
    c.full_reset()                                               # state_output_setup: the filters start again (src/cassiemujoco.c:2032)
    again = _filtered(c.step_pd(pu))
    assert again[8] == pytest.approx(31 * 9.806, rel=1e-6) and np.abs(again[3:6]).max() < 0.05 and 0.4 < again[2] < 1.0


def test_batch_filters_follow_each_environment():
    P = product()
    n = 4
    b0 = P.CassieBatch(1, precision=P.FP64)
    pin1 = (P.pd_in_t * 1)(_pd(P))
    y0 = b0.step_pd(pin1)
    # cassie_sim_step_pd_batch is output-equivalent to cassie_sim_step_pd: the in-kernel estimator comes on with the first call ...
    assert y0[0].pelvis.externalForce[2] == pytest.approx(31 * 9.806, rel=1e-3) and y0[0].pelvis.position[2] != 0
    b0.enable_estimator_device(False)      # ... unless the caller opts out: the filtered fields and the leg forces are then zero
    y0 = b0.step_pd(pin1)
    assert not any(y0[0].pelvis.position[:]) and not any(y0[0].pelvis.externalForce[:]) and not any(y0[0].leftFoot.toeForce[:])
    b = P.CassieBatch(n, precision=P.FP64)
    pin = (P.pd_in_t * n)(*[_pd(P) for _ in range(n)])
    b.enable_estimator()                   # the host-side checker (one filter object per environment); the kernel stage stays off
    c = P.CassieSim()                       # runs the in-kernel estimator
    for k in range(300):
        ys = b.step_pd(pin)
        yc = c.step_pd(pin[0])
        if k == 150:
            m = np.zeros(n, dtype=np.uint8)
            m[2] = 1
            b.reset_estimator(m)
    want = _filtered(yc)
    for e in (0, 1, 3):     # the single-environment object runs the extended kernel instance: equal physics to rounding, not bitwise
        assert (np.abs(_filtered(ys[e]) - want) / (1 + np.abs(want))).max() < 1e-6, e
    assert np.array_equal(_filtered(ys[0]), _filtered(ys[1]))
    assert (np.abs(_filtered(ys[2]) - want) / (1 + np.abs(want))).max() > 1e-3   # environment 2 restarted its filters at call 150


def test_turn_invariance_at_full_size():
    """BASELINE config 2 size, fp64: every environment starts from the same sliding touch-down turned about the vertical by a multiple of 90
    degrees; turned back, all trajectories coincide (exactly the symmetry group of the friction pyramid; CPU twin of this property for the
    oracle and the kernel source: tests/test_oracle.py::test_half_and_quarter_turn_invariance)"""
    P = product()
    n = 4096
    b = P.CassieBatch(n, precision=P.FP64)
    q, v = b.qpos(), b.qvel()
    k = np.arange(n) % 4
    yaw = k * (np.pi / 2)
    c, s = np.round(np.cos(yaw)), np.round(np.sin(yaw))                       # exact quarter turns
    p0, v0 = np.array([0.3, -0.2]), np.array([0.4, 0.1])
    q[:, 0], q[:, 1] = c * p0[0] - s * p0[1], s * p0[0] + c * p0[1]
    v[:, 0], v[:, 1] = c * v0[0] - s * v0[1], s * v0[0] + c * v0[1]
    qz = np.stack([np.cos(yaw / 2), 0 * yaw, 0 * yaw, np.sin(yaw / 2)], axis=1)

    def qmul(a, r):
        return np.stack([a[:, 0] * r[:, 0] - a[:, 1] * r[:, 1] - a[:, 2] * r[:, 2] - a[:, 3] * r[:, 3], a[:, 0] * r[:, 1] + a[:, 1] * r[:, 0] + a[:, 2] * r[:, 3] - a[:, 3] * r[:, 2],
                         a[:, 0] * r[:, 2] - a[:, 1] * r[:, 3] + a[:, 2] * r[:, 0] + a[:, 3] * r[:, 1], a[:, 0] * r[:, 3] + a[:, 1] * r[:, 2] - a[:, 2] * r[:, 1] + a[:, 3] * r[:, 0]], axis=1)
    q[:, 3:7] = qmul(qz, q[:, 3:7])
    b.set_qpos(q)
    b.set_qvel(v)
    b.forward()
    b.set_pd(P.pd_rows(n, pTarget=PD_TARGET, pGain=PD_PGAIN, dGain=PD_DGAIN))
    b.step(400)
    q = b.qpos()
    x, y = q[:, 0].copy(), q[:, 1].copy()
    q[:, 0], q[:, 1] = c * x + s * y, -s * x + c * y                          # turned back
    q[:, 3:7] = qmul(qz * [1, 1, 1, -1], q[:, 3:7])
    ref = q[0]
    assert abs(ref[0] - 0.3) > 0.01 and (b.counters()[:, 1] >= 2).all()       # it landed and slid, everywhere
    for kk, tol in ((0, 0.0), (2, 1e-10), (1, 1e-6), (3, 1e-6)):              # same heading: bitwise; half turn: rounding; quarter turns: row-order noise
        d = np.abs(q[k == kk] - ref).max()
        assert d <= tol, (kk, d)


def test_in_kernel_estimator_rows():
    """the estimator inside the step kernel: rows equal the host-side filters of the one-tick AoS path, and stay exact over multi-tick launches"""
    P = product()
    n = 3
    a, b = P.CassieBatch(n, precision=P.FP64), P.CassieBatch(n, precision=P.FP64)
    pin = (P.pd_in_t * n)(*[_pd(P) for _ in range(n)])
    rows = P.pd_rows(n, pTarget=PD_TARGET, pGain=PD_PGAIN, dGain=PD_DGAIN)
    a.enable_estimator()                       # host filters
    b.enable_estimator_device()                # kernel stage
    b.set_pd(rows)
    for k in range(60):
        for _ in range(5):
            ys = a.step_pd(pin)
        b.step(5)                              # five ticks per launch
    want = np.concatenate([_filtered(ys[1]), ys[1].leftFoot.toeForce[:], ys[1].rightFoot.toeForce[:]])
    got = b.estimator()[1]
    assert (np.abs(got - want) / (1 + np.abs(want))).max() < 1e-8, (got, want)
    m = np.zeros(n, dtype=np.uint8)
    m[0] = 1
    b.reset_estimator(m)
    b.step(1)
    r = b.estimator()
    assert r[0, 8] == pytest.approx(31 * 9.806, rel=1e-6) and abs(r[1, 8] - 31 * 9.806) > 1
