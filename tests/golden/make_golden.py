#!/usr/bin/env python3
"""Regenerates the committed fixtures under tests/golden/ from the reference checkout.
Runs ONLY in the build container (needs /root/reference); the GPU box uses the committed files.

  *.omodel   oracle model tables: oracle/mjcf_compile.py applied to /root/reference/model/<name>.xml
             (derived numeric tables, not a copy of the XML)
  estimator_sequence.npz   400 consecutive 2 kHz calls of the reference's closed estimator (state_output_step) in a closed-loop run from the
             initial state (free fall, touch-down, load transfer): its stateless outputs that feed its filters, and the filters' outputs
  agility_vectors.npz   input/output pairs of the reference's closed Agility blocks (pd_input_step incl. taskPd, cassie_core_sim_step,
             state_output_step from src/libagilitycassie.a via oracle/_ref/liboracle_ref.so; layout: oracle/probe_estimator.c)
  reference_bus_layout.json   the reference's bus struct layout (field lists of its ctypes mirror, gcc offsets from its headers)
  archive_runs.npz   the same blocks in closed loops of the oracle's simulator (sampled records), on the fuzz inputs of oracle/fuzz_agility.c's
             kind and on random estimator inputs: what the twin, controller and estimator tests compare against (archive_runs below)
"""
import os
import sys
HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(REPO, 'oracle'))
import mjcf_compile as mc  # noqa: E402

REF = os.environ.get('CASSIE_REFERENCE', '/root/reference')
MODELS = ['cassie', 'cassie_hfield', 'cassie_tray_box', 'cassie_no_grav', 'cassie_mass', 'cassie_depth']


def agility_vectors(n=400, seed=123):
    """random cassie_out / pd_in_t inputs -> outputs of the REAL closed blocks (src/libagilitycassie.a through oracle/_ref/liboracle_ref.so)"""
    import ctypes as C
    import subprocess
    import numpy as np
    subprocess.check_call(['make', '-s', '-C', os.path.join(REPO, 'oracle'), 'ref', 'REF=' + REF])
    L = C.CDLL(os.path.join(REPO, 'oracle', '_ref', 'liboracle_ref.so'))
    dp = C.POINTER(C.c_double)
    L.probe_est.argtypes = [dp, C.c_int, dp]
    L.probe_pd.argtypes = [dp, dp, C.c_int, dp]
    L.probe_core.argtypes = [dp, dp, C.c_double, dp]
    rng = np.random.default_rng(seed)
    lo, hi = np.array([-0.3, -0.4, -0.9, -2.9, -2.5] * 2), np.array([0.4, 0.4, 1.4, -0.6, -0.5] * 2)
    X, T, U, CH, EST, PD, CORE = [], [], [], [], [], [], []
    for i in range(n):
        x = np.zeros(45)
        x[0:10] = rng.uniform(lo, hi) if i % 4 else rng.uniform(-3, 3, 10)
        x[10:20] = rng.uniform(-8, 8, 10)
        x[20:26] = [rng.uniform(-0.2, 0.2), rng.uniform(0.8, 2.6), rng.uniform(-2.4, -0.6)] * 2
        if i % 2:   # every other sample inside the leg's working range (small spring deflections): what the toe / heel force model is pinned on
            x[0:10] = rng.uniform(np.array([-0.2, -0.3, -0.6, -2.2, -2.2] * 2), np.array([0.3, 0.3, 1.0, -0.9, -0.8] * 2))
            for sd in range(2):
                x[20 + 3 * sd] = rng.uniform(-0.05, 0.05)
                x[21 + 3 * sd] = np.deg2rad(13) - x[5 * sd + 3] - x[20 + 3 * sd] + rng.uniform(-0.05, 0.05)
        x[26:32] = rng.uniform(-6, 6, 6)
        q = rng.normal(size=4)
        x[32:36] = q / np.linalg.norm(q)
        x[36:39], x[39:42] = rng.uniform(-3, 3, 3), rng.uniform(-12, 12, 3)
        t = np.zeros(60)
        if i % 3:
            t[:] = np.concatenate([np.concatenate([rng.uniform(-30, 30, 6), rng.uniform(-1, 1, 6), rng.uniform(-2, 2, 6), rng.uniform(0, 300, 6), rng.uniform(0, 10, 6)]) for _ in range(2)])
        u, ch = rng.uniform(-250, 250, 10), (1.0 if i % 7 else 0.0)
        e, p, c = np.zeros(123), np.zeros(10), np.zeros(10)
        L.probe_est(x.ctypes.data_as(dp), 1, e.ctypes.data_as(dp))
        L.probe_pd(x.ctypes.data_as(dp), t.ctypes.data_as(dp), 1, p.ctypes.data_as(dp))
        L.probe_core(x.ctypes.data_as(dp), u.ctypes.data_as(dp), ch, c.ctypes.data_as(dp))
        X.append(x); T.append(t); U.append(u); CH.append(ch); EST.append(e[:105]); PD.append(p); CORE.append(c)
    np.savez_compressed(os.path.join(HERE, 'agility_vectors.npz'), cassie_out=np.array(X), task=np.array(T), u=np.array(U), ch8=np.array(CH),
                        state_out=np.array(EST), pd_torque=np.array(PD), core_torque=np.array(CORE))
    print('wrote agility_vectors.npz', n)


def estimator_sequence(T=400):
    """closed loop of the oracle's simulator with the REAL closed blocks (oracle/_ref/liboracle_ref.so): per call the archive's own stateless
    outputs the filters consume (orientation 4, translationalAcceleration 3, foot positions 2x3, toe+heel force 2x3 = 19) and the filter
    outputs (position 3, translationalVelocity 3, externalForce 3, terrain.height = 10)"""
    import ctypes as C
    import importlib
    import numpy as np
    sys.path.insert(0, REPO)
    sys.path.insert(0, os.path.join(REPO, 'tests'))
    import oracle as O
    from conftest import PD_DGAIN, PD_PGAIN, PD_TARGET
    pkg = importlib.import_module('cassie-mujoco-sim_b200')
    O.build(ref=True)
    o = O.OracleSim(os.path.join(HERE, 'cassie.omodel'), ref=True)
    u = O.make_pd(pTarget=PD_TARGET, pGain=PD_PGAIN, dGain=PD_DGAIN)
    y = pkg.state_out_t()
    X, Y = [], []
    for k in range(T):
        o.step_pd(u, y)
        X.append(np.concatenate([y.pelvis.orientation[:], y.pelvis.translationalAcceleration[:], y.leftFoot.position[:], y.rightFoot.position[:],
                                 np.array(y.leftFoot.toeForce[:]) + np.array(y.leftFoot.heelForce[:]), np.array(y.rightFoot.toeForce[:]) + np.array(y.rightFoot.heelForce[:])]))
        Y.append(np.concatenate([y.pelvis.position[:], y.pelvis.translationalVelocity[:], y.pelvis.externalForce[:], [y.terrain.height]]))
        assert not any(y.pelvis.externalMoment[:]) and not any(y.terrain.slope[:])
    np.savez_compressed(os.path.join(HERE, 'estimator_sequence.npz'), stateless=np.array(X), filtered=np.array(Y))
    print('wrote estimator_sequence.npz', T)


def archive_runs(every=50, n_fuzz=100, n_random=150):
    """what tests/test_agility_twins.py, tests/test_estimator_filter.py and the GPU estimator tests compare against, from the REAL closed blocks
    (oracle/_ref/liboracle_ref.so):
      <run>_tick / _cassie_out / _state_out / _qpos   closed loops of the oracle's simulator with the real blocks, sampled every `every` ticks:
             the cassie_out_t record and the state_out_t the block made of it (raw struct bytes) and qpos.  Runs: 'pd' = the fixed motor-PD
             controller from the initial state (1200 ticks), 'zero' = zero pd_in_t (1000 ticks), 'spin' = the fixed PD from a spinning attitude
             stored with w < 0 (700 ticks)
      fuzz<mode>_pd / _core   pd_input_step and cassie_core_sim_step on the first n_fuzz inputs of test_agility_twins.fuzz_inputs(mode)
      est_random_feet   the foot outputs (state_out_t flattened [22:35] and [41:54]) on the first n_random inputs of test_agility_twins.random_foot_inputs()
      est_kinematics_feet   the foot positions ([22:25] and [41:44]) on the inputs of test_agility_twins.kinematics_inputs()"""
    import ctypes as C
    import importlib
    import numpy as np
    sys.path.insert(0, REPO)
    sys.path.insert(0, os.path.join(REPO, 'tests'))
    import oracle as O
    import test_agility_twins as T
    from conftest import PD_DGAIN, PD_PGAIN, PD_TARGET
    pkg = importlib.import_module('cassie-mujoco-sim_b200')
    O.build(ref=True)
    out = {}
    fixed = O.make_pd(pTarget=PD_TARGET, pGain=PD_PGAIN, dGain=PD_DGAIN)
    for name, u, spin, ticks in (('pd', fixed, False, 1200), ('zero', O.make_pd(), False, 1000), ('spin', fixed, True, 700)):
        o = O.OracleSim(os.path.join(HERE, 'cassie.omodel'), ref=True)
        if spin:
            T.spin_setup(o)
        y, co = pkg.state_out_t(), (C.c_char * 1336)()
        rows = []
        for k in range(ticks):
            o.step_pd(u, y, co)
            if (k + 1) % every == 0:
                rows.append((k, np.frombuffer(bytes(co), np.uint8), np.frombuffer(bytes(y), np.uint8), o.arr('qpos').copy()))
        for i, key in enumerate(('tick', 'cassie_out', 'state_out', 'qpos')):
            out[name + '_' + key] = np.array([r[i] for r in rows])
    L = O.load(ref=True)
    dp = C.POINTER(C.c_double)
    L.probe_pd_core.argtypes = [dp, C.c_void_p, C.c_double, dp, dp]
    L.probe_est.argtypes = [dp, C.c_int, dp]
    for mode in (0, 1):
        pd, core = np.zeros((n_fuzz, 10)), np.zeros((n_fuzz, 10))
        for i, (x, ch8, u) in enumerate(T.fuzz_inputs(mode, n_fuzz, pkg)):
            L.probe_pd_core(x.ctypes.data_as(dp), C.byref(u), ch8, pd[i].ctypes.data_as(dp), core[i].ctypes.data_as(dp))
        out['fuzz%d_pd' % mode], out['fuzz%d_core' % mode] = pd, core

    def est(x):
        e = np.zeros(123)
        L.probe_est(np.ascontiguousarray(x).ctypes.data_as(dp), 1, e.ctypes.data_as(dp))
        return e
    out['est_random_feet'] = np.array([np.concatenate([e[22:35], e[41:54]]) for e in map(est, T.random_foot_inputs(n_random))])
    out['est_kinematics_feet'] = np.array([np.concatenate([e[22:25], e[41:44]]) for e in map(est, (x for x, _ in T.kinematics_inputs()))])
    np.savez_compressed(os.path.join(HERE, 'archive_runs.npz'), **out)
    print('wrote archive_runs.npz', {k: v.shape for k, v in out.items()})


def bus_layout():
    """reference_bus_layout.json: the bus structs' field lists in the reference's generated ctypes mirror (example/cassiemujoco_ctypes.py) and
    the sizes / offsets gcc gives them from the reference's headers (the probes of tests/test_abi.py)"""
    import json
    import pathlib
    import re
    import tempfile
    sys.path.insert(0, os.path.join(REPO, 'tests'))
    import test_abi
    txt = open(os.path.join(REF, 'example', 'cassiemujoco_ctypes.py')).read()
    fields = {}
    for struct in ('struct_c__SA_pd_in_t', 'struct_c__SA_state_out_t', 'struct_c__SA_state_pelvis_out_t'):
        m = re.search(struct + r'\._fields_ = \[(.*?)\]\n', txt, flags=re.S) or re.search(r'class ' + struct + r'\(.*?_fields_ = \[(.*?)\]\n', txt, flags=re.S)
        fields[struct] = [f for f in re.findall(r"\('(\w+)'", m.group(1)) if not f.startswith('PADDING')]
    with tempfile.TemporaryDirectory() as d:
        offsets = test_abi.bus_offsets(pathlib.Path(d), 'ref', ['pd_in_t.h', 'state_out_t.h', 'cassie_out_t.h', 'cassie_in_t.h', 'cassie_user_in_t.h'],
                                       os.path.join(REF, 'include'))
    with open(os.path.join(HERE, 'reference_bus_layout.json'), 'w') as f:
        json.dump({'ctypes_fields': fields, 'offsets': offsets}, f, indent=1)
        f.write('\n')
    print('wrote reference_bus_layout.json')


def main():
    bus_layout()
    agility_vectors()
    estimator_sequence()
    archive_runs()
    for name in MODELS:
        m = mc.compile_mjcf(os.path.join(REF, 'model', name + '.xml'))
        mc.write_omodel(m, os.path.join(HERE, name + '.omodel'))
        print('wrote', name + '.omodel')


if __name__ == '__main__':
    main()
