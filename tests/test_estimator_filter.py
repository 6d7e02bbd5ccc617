"""The estimator's filters (pelvis.position / translationalVelocity / externalForce, terrain.height of state_out_t; SURVEY.md 8f-1).
Three implementations are compared: the reference's closed block (its committed outputs tests/golden/estimator_sequence.npz and
archive_runs.npz), the oracle's restatement (oracle/cassie_oracle.c o_est_filter_step) and the product's host object
(csrc/estimator_host.h EstimatorFilter through cassie_b200_estimator_filter_step).  No GPU involved."""
import ctypes as C
import os

import numpy as np

from conftest import GOLDEN, PD_DGAIN, PD_PGAIN, PD_TARGET


def _filtered(y):
    return np.concatenate([y.pelvis.position[:], y.pelvis.translationalVelocity[:], y.pelvis.externalForce[:], [y.terrain.height]])


def _load_stateless(y, x):
    """x: orientation 4, translationalAcceleration 3, foot positions 2x3, leg force (toe + heel) 2x3"""
    y.pelvis.orientation[:] = list(x[0:4])
    y.pelvis.translationalAcceleration[:] = list(x[4:7])
    y.leftFoot.position[:] = list(x[7:10])
    y.rightFoot.position[:] = list(x[10:13])
    for f, v in ((y.leftFoot, x[13:16]), (y.rightFoot, x[16:19])):
        f.toeForce[:] = list(0.5 * v)
        f.heelForce[:] = list(0.5 * v)


def _oracle_filter(O):
    L = O.load()
    L.o_est_new.restype = C.c_void_p
    L.o_est_free.argtypes = [C.c_void_p]
    L.o_est_filter_step.argtypes = [C.c_void_p, C.c_void_p]
    L.o_est_filter_reset.argtypes = [C.c_void_p]
    return L


def _product_filter(pkg):
    L = pkg.lib()
    L.cassie_b200_estimator_filter_new.restype = C.c_void_p
    L.cassie_b200_estimator_filter_free.argtypes = [C.c_void_p]
    L.cassie_b200_estimator_filter_reset.argtypes = [C.c_void_p]
    L.cassie_b200_estimator_filter_step.argtypes = [C.c_void_p, C.c_void_p]
    return L


def _rel(a, b):
    return np.abs(a - b) / (1.0 + np.abs(b))


def test_filters_reproduce_the_committed_archive_sequence(oracle_mod, pkg):
    """400 consecutive calls of the closed block (free fall, touch-down at call ~100, the 50 N switch of the foot process noise at call 112):
    oracle and product filters, fed the block's own stateless outputs, give its filtered outputs"""
    V = np.load(os.path.join(GOLDEN, 'estimator_sequence.npz'))
    Lo, Lp = _oracle_filter(oracle_mod), _product_filter(pkg)
    eo, ep = Lo.o_est_new(), Lp.cassie_b200_estimator_filter_new()
    yo, yp = pkg.state_out_t(), pkg.state_out_t()
    worst = np.zeros(2)
    assert V['stateless'][:, 15].min() < -50 < V['stateless'][:50, 15].max()          # both noise regimes are in the sequence
    for x, want in zip(V['stateless'], V['filtered']):
        for y in (yo, yp):
            _load_stateless(y, x)
        Lo.o_est_filter_step(eo, C.byref(yo))
        Lp.cassie_b200_estimator_filter_step(ep, C.byref(yp))
        worst = np.maximum(worst, [_rel(_filtered(yo), want).max(), _rel(_filtered(yp), want).max()])
    Lo.o_est_free(eo)
    Lp.cassie_b200_estimator_filter_free(ep)
    assert worst.max() < 1e-10, worst


def test_product_filter_equals_oracle_filter_on_random_sequences(oracle_mod, pkg):
    """contact making and breaking, both noise regimes, rotated pelvis, restart in the middle"""
    Lo, Lp = _oracle_filter(oracle_mod), _product_filter(pkg)
    rng = np.random.default_rng(11)
    yo, yp = pkg.state_out_t(), pkg.state_out_t()
    worst, seen_contact, seen_air = 0.0, 0, 0
    for trial in range(6):
        eo, ep = Lo.o_est_new(), Lp.cassie_b200_estimator_filter_new()
        q = rng.normal(size=4) * [1, 0.2, 0.2, 0.6]
        q[0] = abs(q[0]) + 1
        foot = np.array([0.0, 0.135, -0.95, 0.0, -0.135, -0.95]) + rng.normal(0, 0.05, 6)
        load = rng.uniform(0, 250, 2)
        for k in range(500):
            q = q + rng.normal(0, 0.002, 4)
            q /= np.linalg.norm(q)
            foot = foot + rng.normal(0, 0.0005, 6)
            phase = np.sin(2 * np.pi * (k / 180.0 + np.array([0.0, 0.5]) + trial / 7.0))
            fz = -np.maximum(0.0, load * phase) * (k % 250 < 170) + rng.normal(0, 0.2, 2)   # stance phases and flights
            force = np.array([rng.normal(0, 20), rng.normal(0, 5), fz[0], rng.normal(0, 20), rng.normal(0, 5), fz[1]])
            x = np.concatenate([q, rng.normal(0, 3, 3) + [0, 0, -9.8 * (k % 2)], foot, force])
            seen_contact += -(min(fz[0], 0) + min(fz[1], 0)) > 1
            seen_air += -(min(fz[0], 0) + min(fz[1], 0)) <= 1
            for y in (yo, yp):
                _load_stateless(y, x)
            if k == 300 and trial % 2:
                Lo.o_est_filter_reset(eo)
                Lp.cassie_b200_estimator_filter_reset(ep)
            Lo.o_est_filter_step(eo, C.byref(yo))
            Lp.cassie_b200_estimator_filter_step(ep, C.byref(yp))
            a, b = _filtered(yo), _filtered(yp)
            assert np.all(np.isfinite(a)) and np.all(np.isfinite(b)), (trial, k)
            worst = max(worst, _rel(b, a).max())
        Lo.o_est_free(eo)
        Lp.cassie_b200_estimator_filter_free(ep)
    assert seen_contact > 500 and seen_air > 500
    assert worst < 1e-9, worst


def test_oracle_estimator_against_live_archive_in_closed_loop(oracle_mod, pkg):
    """the whole restated estimator (stateless part + filters) in a closed-loop run of 1200 calls beside the closed block's outputs on the same run
    (tests/golden/archive_runs.npz, every 50th call); the filters alone, fed the block's own stateless outputs (its 400-call sequence), to
    rounding.  End to end the leg forces limit the agreement (the block evaluates them in single precision)."""
    O = oracle_mod
    L = O.load()
    L.o_est_new.restype = C.c_void_p
    L.o_est_free.argtypes = [C.c_void_p]
    L.o_est_filter_step.argtypes = [C.c_void_p, C.c_void_p]
    L.o_state_output_step_full.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    V, S = np.load(os.path.join(GOLDEN, 'archive_runs.npz')), np.load(os.path.join(GOLDEN, 'estimator_sequence.npz'))
    o = O.OracleSim(os.path.join(GOLDEN, 'cassie.omodel'))
    u = O.make_pd(pTarget=PD_TARGET, pGain=PD_PGAIN, dGain=PD_DGAIN)
    y, y3, y4, co = pkg.state_out_t(), pkg.state_out_t(), pkg.state_out_t(), (C.c_char * 1336)()
    e1, e2 = L.o_est_new(), L.o_est_new()
    err_filter, err_full = 0.0, 0.0
    for x, want in zip(S['stateless'], S['filtered']):
        _load_stateless(y3, x)
        L.o_est_filter_step(e1, C.byref(y3))
        err_filter = max(err_filter, _rel(_filtered(y3), want).max())
    ticks = list(V['pd_tick'])
    for k in range(ticks[-1] + 1):
        o.step_pd(u, y, co)
        L.o_state_output_step_full(e2, C.byref(co), C.byref(y4))
        if k in ticks:
            ya = pkg.state_out_t.from_buffer_copy(V['pd_state_out'][ticks.index(k)].tobytes())     # the archive's state_out_t for this call
            want = _filtered(ya)
            err_full = max(err_full, _rel(_filtered(y4), want).max())
            assert not any(ya.pelvis.externalMoment[:]) and not any(ya.terrain.slope[:])     # never written by the block
    L.o_est_free(e1)
    L.o_est_free(e2)
    assert abs(want[8]) > 1 and abs(want[2]) > 0.3
    assert err_filter < 1e-10 and err_full < 1e-3, (err_filter, err_full)


def test_first_call_against_committed_archive_vectors(oracle_mod, pkg):
    """tests/golden/agility_vectors.npz: a fresh closed block called once on 400 random inputs; the restated estimator's first call (filter start
    included) gives the same pelvis.position / translationalVelocity / externalForce"""
    V = np.load(os.path.join(GOLDEN, 'agility_vectors.npz'))
    L = oracle_mod.load()
    dp = C.POINTER(C.c_double)
    L.osim_fill_cassie_out.argtypes = [C.c_void_p, dp]
    L.o_est_new.restype = C.c_void_p
    L.o_est_free.argtypes = [C.c_void_p]
    L.o_est_filter_reset.argtypes = [C.c_void_p]
    L.o_state_output_step_full.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    e = L.o_est_new()
    y = pkg.state_out_t()
    checked, worst = 0, 0.0
    for x, est in zip(V['cassie_out'], V['state_out']):
        fl, fr = est[37] + est[40], est[56] + est[59]
        if min(abs(fl + 50), abs(fr + 50), abs(min(fl, 0) + min(fr, 0) + 1)) < 0.5 or max(abs(fl), abs(fr)) > 2000:
            continue                                          # next to a switch the single-precision forces decide; implausible loads
        co = (C.c_char * 1336)()
        xx = np.ascontiguousarray(x)
        L.osim_fill_cassie_out(co, xx.ctypes.data_as(dp))
        L.o_est_filter_reset(e)
        L.o_state_output_step_full(e, co, C.byref(y))
        mine = np.array([2 * y.leftFoot.toeForce[2], 2 * y.rightFoot.toeForce[2]])
        if np.any(np.abs(mine - [fl, fr]) > 2e-2 + 2e-4 * np.abs([fl, fr])):
            continue                                          # outside the leg's working range the force model is not pinned (test_agility_twins.py)
        want = np.concatenate([est[0:3], est[10:13], est[19:22], [est[60]]])
        worst = max(worst, _rel(_filtered(y), want).max())
        checked += 1
    L.o_est_free(e)
    assert checked > 150 and worst < 2e-5, (checked, worst)
