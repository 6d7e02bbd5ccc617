"""The closed Agility blocks (pd_input_step motor branch, cassie_core_sim_step): twins vs the reference's archive."""
import os

import numpy as np
import pytest

from conftest import GOLDEN, PD_DGAIN, PD_PGAIN, PD_TARGET, REPO

ARCHIVE_RUNS = os.path.join(GOLDEN, 'archive_runs.npz')   # outputs of the REAL closed blocks (tests/golden/make_golden.py archive_runs)


def archive_runs():
    return np.load(ARCHIVE_RUNS)


def fuzz_inputs(mode, n, pkg, seed=12345):
    """the inputs oracle/fuzz_agility.c draws: drive angles inside the joint ranges (mode 0: mostly well inside, a quarter of them anywhere in
    range; mode 1: anywhere), radio channel 8 random on every 17th input, random motor PD and, on two thirds of the inputs, random task PD.
    Yields (cassie_out as the 45 numbers of oracle/probe_estimator.c, radio channel 8, pd_in_t)."""
    rng = np.random.default_rng(seed + mode)
    lo, hi = np.array([-0.3, -0.4, -0.9, -2.9, -2.5] * 2), np.array([0.3, 0.4, 1.4, -0.6, -0.5] * 2)
    for it in range(n):
        x = np.zeros(45)
        x[32] = 1
        w = np.where((mode == 1) | (rng.random(10) < 0.25), 1.0, 0.55)
        x[0:10] = 0.5 * (lo + hi) + 0.5 * (hi - lo) * w * rng.uniform(-1, 1, 10)
        x[5] = -x[5]
        x[10:20] = rng.uniform(-8, 8, 10)
        x[20:26] = rng.uniform([-0.2, 0.8, -2.4] * 2, [0.2, 2.6, -0.6] * 2)
        x[26:32] = rng.uniform(-6, 6, 6)
        ch8 = rng.uniform(-1, 1) if it % 17 == 0 else 1.0
        u = pkg.pd_in_t()
        for sd, leg in enumerate((u.leftLeg, u.rightLeg)):
            m = rng.uniform([-50, -2, -3, 0, 0], [50, 2, 3, 200, 10], (5, 5))
            for k in range(5):
                leg.motorPd.torque[k], leg.motorPd.pTarget[k], leg.motorPd.dTarget[k], leg.motorPd.pGain[k], leg.motorPd.dGain[k] = m[k]
            if it % 3:
                t = rng.uniform([-30, -1, -2, 0, 0], [30, 1, 2, 300, 10], (6, 5)) * (rng.random((6, 5)) < [1, 1, 1, 0.75, 0.75])
                for k in range(6):
                    leg.taskPd.torque[k], leg.taskPd.pTarget[k], leg.taskPd.dTarget[k], leg.taskPd.pGain[k], leg.taskPd.dGain[k] = t[k]
        yield x, ch8, u


@pytest.mark.parametrize('mode', [0, 1])
def test_oracle_twins_match_archive_on_fuzz(mode, oracle_mod, pkg):
    import ctypes as C
    V = archive_runs()
    L = oracle_mod.load()
    dp = C.POINTER(C.c_double)
    L.osim_fill_cassie_out.argtypes = [C.c_void_p, dp]
    L.o_pd_input_step.argtypes = [C.c_void_p, C.c_void_p, dp]
    L.o_core_sim_step.argtypes = [dp, C.c_void_p, dp]
    want_pd, want_core = V['fuzz%d_pd' % mode], V['fuzz%d_core' % mode]
    err_pd, err_core = 0.0, 0.0
    for (x, ch8, u), pdq, core in zip(fuzz_inputs(mode, len(want_pd), pkg), want_pd, want_core):
        co = (C.c_char * 1336)()
        L.osim_fill_cassie_out(co, np.ascontiguousarray(x).ctypes.data_as(dp))
        L.osim_set_radio8(co, C.c_double(ch8))
        tq, out = (C.c_double * 10)(), (C.c_double * 10)()
        L.o_pd_input_step(C.byref(u), co, tq)
        L.o_core_sim_step(np.ascontiguousarray(pdq).ctypes.data_as(dp), co, out)    # fed the archive's own pd_input_step output, as the fuzz does
        err_pd, err_core = max(err_pd, np.abs(np.array(tq[:]) - pdq).max()), max(err_core, np.abs(np.array(out[:]) - core).max())
    assert len(want_pd) >= 100 and np.abs(want_core).max() > 100
    assert err_pd <= 1e-9 and err_core <= 1e-9, (err_pd, err_core)   # torques up to ~1e4 N m with the fuzzed task gains


def test_product_controller_matches_archive_in_closed_loop(oracle_mod):
    """the product's controller stage (step_core.inl, run through the host emulation in fp64) against the oracle linked with the
    REAL archive blocks, over BASELINE config 1 (zero pd_in_t, 1000 ticks: the collapsing robot drives joints into the safety
    layer's soft limits) and the fixed-PD controller; the archive's trajectory is stored every 50 ticks"""
    import emu_harness as E
    V = archive_runs()
    for run, pd in (('zero', np.zeros(50)), ('pd', np.concatenate([np.zeros(10), PD_TARGET, np.zeros(10), PD_PGAIN, PD_DGAIN]))):
        e = E.EmuSim(os.path.join(REPO, 'cassie-mujoco-sim_b200', 'models', 'cassie.cmodel'))
        ticks, want = list(V[run + '_tick']), V[run + '_qpos']
        worst, safety = 0.0, 0
        for k in range(ticks[-1] + 1):
            e.step(pd)
            safety += e.get('qpos')[14] < -2.5727
            if k in ticks:
                worst = max(worst, np.abs(e.get('qpos')[:35] - want[ticks.index(k)]).max())
        assert worst < 1e-9, (run, worst)
        if not pd.any():
            assert safety > 50     # the safety layer really was exercised


DECODED = ['pelvis.orientation', 'pelvis.rotationalVelocity', 'pelvis.translationalAcceleration', 'leftFoot.position', 'leftFoot.orientation',
           'leftFoot.footRotationalVelocity', 'leftFoot.footTranslationalVelocity', 'rightFoot.position', 'rightFoot.orientation',
           'rightFoot.footRotationalVelocity', 'rightFoot.footTranslationalVelocity', 'motor.position', 'motor.velocity', 'motor.torque',
           'joint.position', 'joint.velocity']


def field(y, path):
    for p in path.split('.'):
        y = getattr(y, p)
    return np.array(y[:])


def spin_setup(o):
    """a spinning attitude stored with w < 0 (the estimator reports the w >= 0 twin)"""
    o.arr('qpos')[3:7] = [-0.995, 0.02, -0.03, 0.09]
    o.arr('qvel')[3:6] = [0.5, -0.4, 0.6]


def test_estimator_twin_matches_archive_in_closed_loop(oracle_mod, pkg):
    """the decoded stateless subset of state_output_step (oracle o_state_output_step) against the REAL estimator, fed the same cassie_out
    along a falling-and-catching trajectory (large joint excursions; an IMU quaternion with w < 0); the archive's records every 50 ticks"""
    import ctypes as C
    V = archive_runs()
    L = oracle_mod.load()
    L.o_state_output_step.argtypes = [C.c_void_p, C.c_void_p]
    worst = {k: 0.0 for k in DECODED}
    for run in ('zero', 'spin'):
        for co, ya in zip(V[run + '_cassie_out'], V[run + '_state_out']):
            y, y2 = pkg.state_out_t.from_buffer_copy(ya.tobytes()), pkg.state_out_t()
            L.o_state_output_step((C.c_char * 1336).from_buffer_copy(co.tobytes()), C.byref(y2))
            for f in DECODED:
                worst[f] = max(worst[f], np.abs(field(y, f) - field(y2, f)).max())
    assert V['spin_qpos'][:, 3].min() < 0
    for f, w in worst.items():
        assert w < 1e-11, (f, w)


def random_foot_inputs(n, seed=11):
    """arbitrary angles / rates, as the 45 cassie_out numbers of oracle/probe_estimator.c"""
    rng = np.random.default_rng(seed)
    for it in range(n):
        x = np.zeros(45)
        x[32] = 1
        x[0:10], x[10:20], x[20:26], x[26:32] = rng.uniform(-3, 3, 10), rng.uniform(-8, 8, 10), rng.uniform(-3, 3, 6), rng.uniform(-8, 8, 6)
        yield x


def kinematics_inputs(n=50, seed=4):
    """random leg configurations inside the joint ranges: (the 45 cassie_out numbers, qpos of the same configuration)"""
    rng = np.random.default_rng(seed)
    lo, hi = np.array([-0.25, -0.35, -0.8, -2.7, -2.4]), np.array([0.3, 0.35, 1.3, -0.7, -0.6])
    for it in range(n):
        mL, mR, sh, ta = rng.uniform(lo, hi), rng.uniform(lo, hi), rng.uniform(-0.05, 0.05, 2), rng.uniform(0.9, 2.0, 2)
        q = np.zeros(35)
        q[2], q[3], q[10], q[24] = 1.01, 1, 1, 1
        q[[7, 8, 9, 14, 20]], q[15], q[16] = mL, sh[0], ta[0]
        q[[21, 22, 23, 28, 34]], q[29], q[30] = mR, sh[1], ta[1]
        x = np.zeros(45)
        x[32] = 1
        x[0:5], x[5:10], x[20], x[21], x[23], x[24] = mL, mR, sh[0], ta[0], sh[1], ta[1]
        yield x, q


def test_estimator_twin_on_random_inputs(oracle_mod):
    """o_est_foot against the archive on arbitrary angles / rates (far outside what a trajectory visits: all mat2quat branches)"""
    import ctypes as C
    want = archive_runs()['est_random_feet']
    L = oracle_mod.load()
    L.o_est_foot.argtypes = [C.c_int] + [C.POINTER(C.c_double)] * 6
    worst = 0.0
    for x, e in zip(random_foot_inputs(len(want)), want):
        for sd in range(2):
            ang = (C.c_double * 7)(*x[5 * sd:5 * sd + 4], x[20 + 3 * sd], x[21 + 3 * sd], x[5 * sd + 4])
            rate = (C.c_double * 7)(*x[10 + 5 * sd:14 + 5 * sd], x[26 + 3 * sd], x[27 + 3 * sd], x[14 + 5 * sd])
            out = [(C.c_double * n)() for n in (3, 4, 3, 3)]
            L.o_est_foot(sd, ang, rate, *out)
            got = np.concatenate([np.array(a[:]) for a in out])
            worst = max(worst, np.abs(got - e[13 * sd:13 * sd + 13]).max())
    assert len(want) >= 150 and worst < 1e-12, worst


def test_archive_kinematics_pin_the_mjcf_compiler(oracle_mod):
    """an independent check of the model compiler's kinematic tables: the foot point computed by the oracle's mj_kinematics on the compiled
    model/cassie.xml equals the closed estimator's own forward kinematics (which carries Agility's constants) to the MJCF's 5-digit rounding"""
    want = archive_runs()['est_kinematics_feet']
    o = oracle_mod.OracleSim(os.path.join(GOLDEN, 'cassie.omodel'))
    names = open(os.path.join(GOLDEN, 'cassie.omodel')).read().split('names_body')[1].split('\n')[0].split()[2:]
    pel, feet = names.index('cassie-pelvis'), (names.index('left-foot'), names.index('right-foot'))
    worst = 0.0
    for (x, q), e in zip(kinematics_inputs(), want):
        o.arr('qpos')[:] = q
        o.forward()
        xp, xm = o.arr('xpos').reshape(-1, 3), o.arr('xmat').reshape(-1, 3, 3)
        for sd, fb in enumerate(feet):
            p = xm[pel].T @ (xp[fb] + xm[fb] @ np.array([0.01762, 0.05219, 0]) - xp[pel])
            worst = max(worst, np.abs(p - e[3 * sd:3 * sd + 3]).max())
    assert len(want) == 50 and worst < 5e-7, worst


def test_twins_against_committed_archive_vectors(oracle_mod, pkg):
    """tests/golden/agility_vectors.npz holds outputs of the REAL closed blocks on 300 random inputs (tests/golden/make_golden.py); the oracle's
    twins reproduce them with no archive present -- this is what pins the twins on the GPU box"""
    import ctypes as C
    V = np.load(os.path.join(GOLDEN, 'agility_vectors.npz'))
    L = oracle_mod.load()
    dp = C.POINTER(C.c_double)
    L.o_est_foot.argtypes = [C.c_int] + [dp] * 6
    L.o_pd_input_step.argtypes = [C.c_void_p, C.c_void_p, dp]
    L.o_core_sim_step.argtypes = [dp, C.c_void_p, dp]
    L.o_state_output_step.argtypes = [C.c_void_p, C.c_void_p]
    # build cassie_out_t / pd_in_t images with ctypes mirrors of the bus structs: use the product's mirrors for pd_in_t and a raw
    # buffer + the oracle's own accessor layout for cassie_out_t (offsets from include/cassie_bus.h via a tiny C helper)
    L.osim_fill_cassie_out.argtypes = [C.c_void_p, dp]
    worst = dict(est=0.0, pd=0.0, core=0.0)
    for x, t, u, ch, est, pdq, core in zip(V['cassie_out'], V['task'], V['u'], V['ch8'], V['state_out'], V['pd_torque'], V['core_torque']):
        co = (C.c_char * 1336)()
        xx = np.ascontiguousarray(x)
        L.osim_fill_cassie_out(co, xx.ctypes.data_as(dp))
        y = pkg.state_out_t()
        L.o_state_output_step(co, C.byref(y))
        got = np.concatenate([[0, 0, 0], field(y, 'pelvis.orientation'), field(y, 'pelvis.rotationalVelocity'), [0, 0, 0], field(y, 'pelvis.translationalAcceleration')])
        want = est[:16].copy()
        want[0:3] = 0
        want[10:13] = 0                                  # pelvis position / translational velocity: the filters, checked in tests/test_estimator_filter.py
        worst['est'] = max(worst['est'], np.abs(got - want).max())
        for sd, name in enumerate(('leftFoot', 'rightFoot')):
            g = np.concatenate([field(y, name + '.position'), field(y, name + '.orientation'), field(y, name + '.footRotationalVelocity'), field(y, name + '.footTranslationalVelocity')])
            worst['est'] = max(worst['est'], np.abs(g - est[22 + 19 * sd:35 + 19 * sd]).max())
        pu = pkg.pd_in_t()
        for sd, leg in enumerate((pu.leftLeg, pu.rightLeg)):
            r = t[30 * sd:30 * sd + 30]
            for k in range(6):
                leg.taskPd.torque[k], leg.taskPd.pTarget[k], leg.taskPd.dTarget[k], leg.taskPd.pGain[k], leg.taskPd.dGain[k] = r[k], r[6 + k], r[12 + k], r[18 + k], r[24 + k]
        tq = (C.c_double * 10)()
        L.o_pd_input_step(C.byref(pu), co, tq)
        worst['pd'] = max(worst['pd'], np.abs(np.array(tq[:]) - pdq).max() / max(1.0, np.abs(pdq).max()))
        co2 = (C.c_char * 1336)()
        L.osim_fill_cassie_out(co2, xx.ctypes.data_as(dp))
        L.osim_set_radio8(co2, C.c_double(float(ch)))
        uu, out = np.ascontiguousarray(u), (C.c_double * 10)()
        L.o_core_sim_step(uu.ctypes.data_as(dp), co2, out)
        worst['core'] = max(worst['core'], np.abs(np.array(out[:]) - core).max())
    assert worst['est'] < 1e-11 and worst['pd'] < 1e-12 and worst['core'] < 1e-9, worst


def test_toe_heel_force_twin(oracle_mod, pkg):
    """toeForce / heelForce: the decoded spring-force model against the real estimator.  The archive evaluates it in single precision, so the
    bar is its own rounding noise (a few mN on forces of ~100 N), not 1e-12: |twin - archive| <= 2e-2 N + 2e-4 |F| in closed loop and on the
    committed random vectors whose deflections are physically plausible"""
    import ctypes as C
    V = np.load(os.path.join(GOLDEN, 'agility_vectors.npz'))
    L = oracle_mod.load()
    dp = C.POINTER(C.c_double)
    L.o_est_leg_force.argtypes = [C.c_int, dp, dp, dp]
    checked = 0
    for x, est in zip(V['cassie_out'], V['state_out']):
        for sd in range(2):
            m, sh, ta = x[5 * sd:5 * sd + 5], x[20 + 3 * sd], x[21 + 3 * sd]
            if abs(sh) > 0.1 or abs(m[3] + sh + ta - np.deg2rad(13)) > 0.1 or not (-2.5 < m[3] < -0.7) or abs(m[0]) > 0.5 or abs(m[1]) > 0.5 or abs(m[2]) > 1.3:
                continue                                    # outside the leg's working range (the four-bar flips, the x-z solve degenerates)
            ang, q, f = (C.c_double * 7)(m[0], m[1], m[2], m[3], sh, ta, m[4]), (C.c_double * 4)(*x[32:36]), (C.c_double * 3)()
            L.o_est_leg_force(sd, ang, q, f)
            want = est[35 + 19 * sd:38 + 19 * sd]
            assert np.abs(np.array(f[:]) - want).max() <= 2e-2 + 2e-4 * np.abs(want).max(), (sd, f[:], want)
            assert np.array_equal(want, est[38 + 19 * sd:41 + 19 * sd])        # the archive reports the same vector for toe and heel
            checked += 1
    V = archive_runs()                                  # closed loop: the archive's records every 50 ticks of the fixed-PD run
    L.o_state_output_step.argtypes = [C.c_void_p, C.c_void_p]
    big = 0.0
    for co, ya in zip(V['pd_cassie_out'], V['pd_state_out']):
        y, y2 = pkg.state_out_t.from_buffer_copy(ya.tobytes()), pkg.state_out_t()
        L.o_state_output_step((C.c_char * 1336).from_buffer_copy(co.tobytes()), C.byref(y2))
        for name in ('leftFoot', 'rightFoot'):
            for fld in ('toeForce', 'heelForce'):
                a, b = field(y, name + '.' + fld), field(y2, name + '.' + fld)
                assert np.abs(a - b).max() <= 2e-2 + 2e-4 * np.abs(a).max(), (name, fld, a, b)
                big = max(big, np.abs(a).max())
    assert big > 30                                           # standing: the springs carry the weight
    checked += 1
    assert checked > 0
