"""GPU: state_out_t filled by cassie_sim_step_pd(_batch) against the REAL estimator archive's outputs (tests/golden/archive_runs.npz) and the oracle, decoded fields."""
import os

import numpy as np
import pytest

from conftest import GOLDEN, PD_DGAIN, PD_PGAIN, PD_TARGET, product
from test_agility_twins import DECODED, field
from test_estimator import row_vs_state_out, row_vs_twin

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def P():
    return product()


def _pd(P):
    pu = P.pd_in_t()
    for side, leg in enumerate((pu.leftLeg, pu.rightLeg)):
        for i in range(5):
            leg.motorPd.pTarget[i] = PD_TARGET[5 * side + i]
            leg.motorPd.pGain[i], leg.motorPd.dGain[i] = PD_PGAIN[i], PD_DGAIN[i]
    return pu


def test_state_out_matches_real_estimator(P, oracle_mod):
    """every call against the oracle's pinned twin of the estimator; every 50th call against the real archive's output on the same run
    (tests/golden/archive_runs.npz)"""
    O = oracle_mod
    V = np.load(os.path.join(GOLDEN, 'archive_runs.npz'))
    ticks = list(V['pd_tick'])
    o = O.OracleSim(os.path.join(GOLDEN, 'cassie.omodel'))
    c = P.CassieSim()
    u, pu, y = O.make_pd(pTarget=PD_TARGET, pGain=PD_PGAIN, dGain=PD_DGAIN), _pd(P), P.state_out_t()
    worst = {k: 0.0 for k in DECODED}
    for k in range(600):
        o.step_pd(u, y)
        yc = c.step_pd(pu)
        refs = [y] + ([P.state_out_t.from_buffer_copy(V['pd_state_out'][ticks.index(k)].tobytes())] if k in ticks else [])
        for yr in refs:
            for f in DECODED:
                worst[f] = max(worst[f], np.abs(field(yr, f) - field(yc, f)).max())
            for name in ('leftFoot', 'rightFoot'):    # toe / heel forces (host-side part, always on for a cassie_sim_t): the archive's single-precision noise is the bar
                for fld in ('toeForce', 'heelForce'):
                    a, b = field(yr, name + '.' + fld), field(yc, name + '.' + fld)
                    assert np.abs(a - b).max() <= 2e-2 + 2e-4 * np.abs(a).max(), (k, name, fld, a, b)
    for f, w in worst.items():
        assert w < 1e-8, (f, w)
    assert abs(yc.leftFoot.position[2] + 0.9) < 0.2 and yc.pelvis.translationalAcceleration[2] != 0
    assert abs(yc.leftFoot.toeForce[2]) > 10


def test_batch_rows_and_aos(P, oracle_mod):
    """the batched AoS entry point and the device observation row carry the same numbers; fp32 rows are self-consistent"""
    n = 5
    b = P.CassieBatch(n, precision=P.FP64)
    pin = (P.pd_in_t * n)(*[_pd(P) for _ in range(n)])
    for _ in range(200):
        ys = b.step_pd(pin)
    rows = b.obs()
    for e in (0, n - 1):
        row_vs_state_out(rows[e], ys[e], 1e-12)
    assert abs(ys[0].leftFoot.toeForce[2]) > 10 and ys[0].leftFoot.toeForce[2] == ys[0].leftFoot.heelForce[2]    # in-kernel estimator: on by default for the AoS entry point
    assert rows[0][P.OBS['est_left_toe_force']][2] == ys[0].leftFoot.toeForce[2] and rows[0][P.OBS['est_position']][2] == ys[0].pelvis.position[2]
    dev = ys[0].leftFoot.toeForce[2]
    P.lib().cassie_batch_enable_estimator_forces(b.h, 1)        # host-side checker of the same function
    ys = b.step_pd(pin)
    assert abs(ys[0].leftFoot.toeForce[2] - dev) < 2e-2 * abs(dev)     # one tick later: the same force up to the robot's motion in 0.5 ms
    b32 = P.CassieBatch(n, precision=P.FP32)
    b32.set_pd(P.pd_rows(n, pTarget=PD_TARGET, pGain=PD_PGAIN, dGain=PD_DGAIN))
    b32.step(300)
    row_vs_twin(oracle_mod, b32.obs()[2], 2e-5)
