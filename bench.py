#!/usr/bin/env python3
"""bench.py -- Cassie env-steps/s for the cassie_sim_step_pd hot path (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--config 2|3|4|5] [--impl reference] [--envs E] [--no-extra] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

One "step" = one control tick (one cassie_sim_step_pd: 0.5 ms of simulated time, 1 physics sub-step) for EVERY environment of the batch.
Workloads (SURVEY.md section 8d, per GPU; N > 1 = the same workload on every GPU, weak scaling, no data-path collective):
  --config 2 (default, the configuration BASELINE.json's metric is quoted on): 4096 envs, cassie.xml flat floor, fixed motor-PD targets
  --config 3: 16384 envs, the same plus pelvis pushes: every 400 ticks xy ~ U(-100, 100) N for 100 ticks, Philox seed 1234 keyed by (env, event)
  --config 4: 8192 envs, cassie_hfield.xml, 64 terrains (seed 7, iid U(0,1) x 0.25 of the 0.2 m elevation scale = 5 cm, flat 10x10 centre patch)
  --config 5: 8192 envs, cassie_tray_box.xml, random PD gaits pTarget(t) = offset + A sin(2 pi f t + phi), f ~ U(0.5, 1.5) Hz, A = (.05,.05,.3,.4,.3),
              left / right phase offset pi, Philox seed 99 (evaluated in the kernel: cassie_batch_set_pd_gait)

value     kernel-only throughput in SINGLE-TICK launches (one cassie_sim_step_pd per launch, the reference's contract): PD rows and state resident
          in HBM, inputs larger than L2 (independent copies of the batch stepped round-robin, > 1.5 x L2 in total).  Exactly K steps are timed,
          as one block with CUDA events on the launching stream; max over ranks.  multi_tick_launches: the same K ticks in launches of T <= 50
          ticks (PD rows held).
e2e       the same metric through the reference-shaped C-ABI call cassie_sim_step_pd_batch(envs, pd_in_t[] host, state_out_t[] host) with the
          WHOLE state_out_t filled as the reference's state_output_step fills it (the estimator runs inside the kernel): host->device copy of
          every env's PD input and device->host read of every env's observation inside the timed region, K steps.
--dump-outputs DIR: after the timed steps, what the last timed step computed, as a caller of the path reads it back (qpos, qvel, time and the
          observation rows of the batch copy that step advanced; rank 0), is written to DIR/<name>.npy in float64.  Inputs are seeded, so two
          builds run with the same arguments can be compared output for output.
roofline  dominant kernel (cassie_step_kernel<float>): HBM figure by the contract's rules (algorithmic state bytes per launch / launch time) and,
          because the kernel is issue / latency bound by design, the issue-slot fraction next to it.
cpu_baseline / --impl reference: the CPU restatement in oracle/ (physics restated from MuJoCo 2.1.0 semantics + the reference's real closed
          Agility blocks when oracle/_ref/liboracle_ref.so exists), one private sim per thread, threads = the CPUs this process may really use
          (affinity mask clipped by the cgroup quota).  The reference's own libcassiemujoco.so cannot be built: no MuJoCo on either machine
          (profiles/r2_probe_reference_*.json).
"""
import argparse
import ctypes as C
import importlib
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, 'oracle'))

PD_TARGET = [0.0045, 0, 0.4973, -1.1997, -1.5968, -0.0045, 0, 0.4973, -1.1997, -1.5968]
PD_PGAIN = [70, 70, 100, 100, 50] * 2
PD_DGAIN = [7, 7, 8, 8, 5] * 2
GAIT_AMP = [0.05, 0.05, 0.3, 0.4, 0.3] * 2
L2_BYTES = 126e6
MIN_TIMED_MS = 100.0

CONFIGS = {
    2: dict(envs=4096, model='cassie', name='config2: 4096 envs/GPU cassie.xml flat floor, fixed motor-PD targets, pelvis z/yaw jitter U(-0.01,0.01) seed 0'),
    3: dict(envs=16384, model='cassie', name='config3: 16384 envs/GPU cassie.xml, fixed motor-PD targets + pelvis pushes every 400 ticks (xy ~ U(-100,100) N held 100 ticks, Philox seed 1234 keyed by env/event)'),
    4: dict(envs=8192, model='cassie_hfield', name='config4: 8192 envs/GPU cassie_hfield.xml, 64 terrains shared round-robin (seed 7, U(0,1) x 0.25 of the 0.2 m scale = 5 cm, flat centre patch), fixed motor-PD targets'),
    5: dict(envs=8192, model='cassie_tray_box', name='config5: 8192 envs/GPU cassie_tray_box.xml (5 kg cup on the pelvis tray), random PD gaits f ~ U(0.5,1.5) Hz, A = (.05,.05,.3,.4,.3) rad, L/R phase offset pi, Philox seed 99'),
}
# warp instructions per env-step and DRAM bytes per launch of the dominant kernel, from the committed ncu capture (static: ncu cannot run inside a
# timed bench).  profiles/r2_step_kernel_counts.json is written by tools/ncu_counts.py from the .ncu-rep the summary next to it was made from.
def _kernel_counts():
    try:
        with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'profiles', 'r2_step_kernel_counts.json')) as f:
            return json.load(f)
    except (OSError, ValueError):
        return {}


KERNEL_COUNTS = _kernel_counts()


# ------------------------------------------------------------------------------ host CPUs
def aos_threads_for_rank(cpus_now, per_rank_share):
    """pack / unpack threads of one rank: its pinned CPUs, never more than its share of the job's CPU quota, at most 32, minus two (kept free for the
    rank's CUDA driver / NCCL / sampler threads: the OpenMP team busy-waits, and teams that add up to the quota get the whole cgroup throttled)"""
    share = min(32, cpus_now, per_rank_share)
    return max(2, share - 2 if share > 4 else share)


def effective_cpus():
    """CPUs this process may really use: affinity mask clipped by the cgroup CPU quota (a 1-GPU lease on a 128-thread host may own 16)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    quota = None
    try:
        q, p = open('/sys/fs/cgroup/cpu.max').read().split()[:2]
        if q != 'max':
            quota = int(q) / int(p)
    except Exception:
        try:
            q = int(open('/sys/fs/cgroup/cpu/cpu.cfs_quota_us').read()); p = int(open('/sys/fs/cgroup/cpu/cpu.cfs_period_us').read())
            if q > 0:
                quota = q / p
        except Exception:
            pass
    eff = n if quota is None else max(1, min(n, int(math.ceil(quota))))
    return eff, n, quota


def pin_rank_to_its_share(local_rank, world):
    """N ranks on one node: give each rank its own slice of the allowed CPUs, on the NUMA node of its GPU when the topology can be read
    (the AoS entry point's pack / unpack threads and its pinned staging buffers then stay next to the GPU's PCIe root)."""
    if world <= 1:
        return None
    try:
        allowed = sorted(os.sched_getaffinity(0))
        node_of = {}
        base = '/sys/devices/system/node'
        for d in os.listdir(base):
            if d.startswith('node') and d[4:].isdigit():
                for part in open(os.path.join(base, d, 'cpulist')).read().strip().split(','):
                    a, _, b = part.partition('-')
                    for c in range(int(a), int(b or a) + 1):
                        node_of[c] = int(d[4:])
        gpu_node = None
        try:
            out = subprocess.run(['nvidia-smi', '-i', str(local_rank), '--query-gpu=pci.bus_id', '--format=csv,noheader'], capture_output=True, text=True, timeout=20).stdout.strip()
            bus = out.lower()
            if bus.startswith('0000'):
                bus = bus[4:]
            gpu_node = int(open('/sys/bus/pci/devices/%s/numa_node' % bus).read())
        except Exception:
            pass
        if gpu_node is not None and gpu_node >= 0 and node_of:
            nodes = sorted(set(node_of.values()))
            per_node = max(1, world // len(nodes))
            mine = [c for c in allowed if node_of.get(c) == gpu_node]
            k = local_rank % per_node
            share = mine[k::per_node] if len(mine) >= per_node else mine
        else:
            share = allowed[local_rank::world]
        if share:
            os.sched_setaffinity(0, share)
            return {'cpus': len(share), 'numa_node': gpu_node}
    except Exception as ex:
        return {'error': repr(ex)}
    return None


def jittered_qpos(q0, n, seed=0):
    rng = np.random.default_rng(seed)
    q = np.repeat(q0[None, :], n, axis=0).copy()
    q[:, 2] += rng.uniform(-0.01, 0.01, n)
    yaw = rng.uniform(-0.01, 0.01, n)
    q[:, 3] = np.cos(yaw / 2); q[:, 4] = 0; q[:, 5] = 0; q[:, 6] = np.sin(yaw / 2)
    return q


def philox_uniform(seed, event, shape, lo, hi):
    """counter-based stream: key = seed, counter word 2 = event; position in the stream = env index, so env e's draw for an event does not
    depend on how many environments the batch has"""
    g = np.random.Generator(np.random.Philox(key=seed, counter=[0, 0, int(event), 0]))
    return g.uniform(lo, hi, shape)


REF_TICKS = 250   # control ticks per reference-arm step


# ------------------------------------------------------------------------------ CPU arm (oracle)
def cpu_arm(n_threads, envs_per_thread, ticks, warm_ticks=0, model='cassie'):
    """aggregate env-steps/s of the CPU oracle with one thread per core, each owning private sims."""
    import oracle as O
    ref = os.path.exists(O.lib_path(ref=True))
    L = O.load(ref=ref)
    mpath = os.path.join(REPO, 'tests', 'golden', model + '.omodel')
    u = O.make_pd(pTarget=PD_TARGET, pGain=PD_PGAIN, dGain=PD_DGAIN)
    groups = []
    for _ in range(n_threads):
        sims = (C.c_void_p * envs_per_thread)(*[L.osim_new(mpath.encode()) for _ in range(envs_per_thread)])
        groups.append(sims)

    def run(sims, t):
        L.osim_run(sims, envs_per_thread, C.byref(u), t)

    def run_all(t):
        th = [threading.Thread(target=run, args=(g, t)) for g in groups]
        t0 = time.perf_counter()
        for x in th:
            x.start()
        for x in th:
            x.join()
        return time.perf_counter() - t0
    if warm_ticks:
        run_all(warm_ticks)
    dt = run_all(ticks)
    for g in groups:
        for s in g:
            L.osim_free(s)
    return n_threads * envs_per_thread * ticks / dt, dt, ref


def cpu_baseline(total_ticks_per_thread, model='cassie'):
    """the oracle at its best thread count: the CPUs this process may use and half of them (hyper-thread pairs), whichever is faster"""
    eff, visible, quota = effective_cpus()
    tried = {}
    best = None
    for nt in sorted({eff, max(1, eff // 2)}, reverse=True):
        val, dt, ref = cpu_arm(nt, 1, total_ticks_per_thread, warm_ticks=300, model=model)
        tried[nt] = val
        if best is None or val > best[0]:
            best = (val, nt, dt, ref)
    val, nt, dt, ref = best
    return {'value': val, 'unit': 'env-steps/s', 'cores': nt, 'kind': 'port', 'per_core': val / nt, 'visible_cpus': visible, 'cgroup_cpu_quota': quota,
            'threads_tried': {str(k): v for k, v in tried.items()},
            'sample': '%d envs (%d threads x 1 private sim) x %d ticks of the same workload on %s; oracle/cassie_oracle.c fp64 + %s' % (
                nt, nt, total_ticks_per_thread, model + '.xml', 'the reference Agility archive (real pd_input_step / cassie_core_sim_step / state_output_step)' if ref else 'Agility twins')}


def reference_arm(args, rank, world):
    if rank != 0:
        return
    cfg = CONFIGS[args.config]
    eff, visible, quota = effective_cpus()
    ticks = REF_TICKS * args.steps
    tried, best = {}, None
    for nt in sorted({eff, max(1, eff // 2)}, reverse=True):
        val, dt, ref = cpu_arm(nt, 1, ticks, warm_ticks=REF_TICKS * min(args.warmup, 2), model=cfg['model'])
        tried[nt] = val
        if best is None or val > best[0]:
            best = (val, nt, dt, ref)
    val, nt, dt, ref = best
    sample = '%d envs (%d threads x 1 private sim) x %d ticks (%d per step) of %s with fixed motor-PD targets; physics = oracle/cassie_oracle.c (fp64 restatement of MuJoCo 2.1.0 semantics, parity unpinned), Agility blocks = %s' % (
        nt, nt, ticks, REF_TICKS, cfg['model'] + '.xml', 'the reference archive libagilitycassie.a incl. state_output_step' if ref else 'oracle twins')
    line = {'impl': 'reference', 'metric': 'Cassie env-steps/s', 'value': val, 'unit': 'env-steps/s', 'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': 1e3 * dt / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
            'config': {'workload': cfg['name'], 'parallelism': 'cpu x%d threads' % nt, 'note': 'one step of this arm = %d control ticks of %d private sims' % (REF_TICKS, nt)},
            'cpu_baseline': {'value': val, 'unit': 'env-steps/s', 'cores': nt, 'kind': 'port', 'per_core': val / nt, 'visible_cpus': visible, 'cgroup_cpu_quota': quota,
                             'threads_tried': {str(k): v for k, v in tried.items()}, 'sample': sample},
            'e2e': {'value': val, 'unit': 'env-steps/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}, 'gpu_launches': 0}
    print(json.dumps(line, default=lambda o: o.tolist() if hasattr(o, 'tolist') else str(o)), flush=True)


# ------------------------------------------------------------------------------ GPU arm
class ClockSampler:
    def __init__(self, gpu_index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(gpu_index), '--query-gpu=clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,'
                                          'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap',
                                          '--format=csv,noheader,nounits', '-lms', '100'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            out = self.proc.communicate(timeout=5)[0]
        except Exception:
            out = ''
        sm, mx, reasons = [], [], set()
        for ln in out.strip().splitlines():
            f = [x.strip() for x in ln.split(',')]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[2:6]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None, 'reasons': sorted(reasons)}


class Workload:
    """one BASELINE configuration on one GPU: builds the batch copies, knows what happens between ticks (pushes), and its byte counts"""

    def __init__(self, P, config, n, device, rank, torch):
        self.P, self.config, self.n, self.device, self.rank, self.torch = P, config, n, device, rank, torch
        self.cfg = CONFIGS[config]
        self.rows = P.pd_rows(n, pTarget=PD_TARGET, pGain=PD_PGAIN, dGain=PD_DGAIN)
        self.own_ticks = {}    # copy index -> control ticks stepped in single-tick launches (the clock of config 3's push schedule)
        self.terrains = None
        if config == 4:
            t = (np.random.default_rng(7).uniform(0, 1, (64, 200, 200)) * 0.25).astype(np.float32)
            t[:, 95:105, 95:105] = 0
            self.terrains = t

    def make_copy(self, k):
        P, n = self.P, self.n
        b = P.CassieBatch(n, modelfile=P.model_path(self.cfg['model']), device=self.device, precision=P.FP32)
        if self.torch is not None:
            b.set_stream(self.torch.cuda.current_stream().cuda_stream)
        if self.terrains is not None:
            b.set_hfield_data(self.terrains)
        q0 = b.qpos()[0]
        q = jittered_qpos(q0, n, seed=1000 * k + self.rank)
        b.set_qpos(q); b.forward(); b.set_pd(self.rows)
        if self.config == 5:
            f = philox_uniform(99, 0, n, 0.5, 1.5); ph = philox_uniform(99, 1, n, 0.0, 2 * np.pi)
            phase = ph[:, None] + np.array([0.0] * 5 + [np.pi] * 5)[None, :]
            b.set_pd_gait(np.array(GAIT_AMP), f, phase)
        return b

    def row_bytes(self, b):
        """state rows read + written per env per single-tick launch (fp32): the algorithmic HBM bytes of the step kernel"""
        qw, vw = b.row_width('qpos'), b.row_width('qvel')
        rd = qw + 2 * vw + 192 + 52 + 8 + 96        # qpos, qvel, warm start, controller state, PD row, xfrc, FIR taps
        wr = qw + 2 * vw + 192 + 96 + self.P.OBS_WIDTH
        return 4 * (rd + wr)

    def footprint(self, b):
        qw, vw = b.row_width('qpos'), b.row_width('qvel')
        return self.n * (qw + 2 * vw + 192 + 52 + 8 + 96 + 2 * 320 + self.P.OBS_WIDTH + 8) * 4

    def before_step(self, b, j, nb):
        """host-driven events of the workload that fall on copy j's next control tick (inside the timed region when they occur).  The copies'
        push schedules are staggered by 400 / nb ticks, so that at any moment the fraction of environments under push is the workload's 25 %."""
        if self.config == 3:
            own = self.own_ticks.setdefault(j, 0)
            t = own + (j * 400) // max(nb, 1)
            ph = t % 400
            if ph == 0:
                push = np.zeros((self.n, 6)); push[:, :2] = philox_uniform(1234, t // 400, (self.n, 2), -100.0, 100.0)
                b.apply_force(push, 'cassie-pelvis')
            elif ph == 100:
                b.clear_forces()
            self.own_ticks[j] = own + 1


def gpu_arm(args, rank, local_rank, world):
    import torch
    P = importlib.import_module('cassie-mujoco-sim_b200')
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    torch.cuda.set_device(local_rank)
    cfg = CONFIGS[args.config]
    n = args.envs or cfg['envs']
    W = Workload(P, args.config, n, local_rank, rank, torch)
    b = W.make_copy(0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(REPO, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    hbm_peak, peak_src = (peaks['hbm_gbs'], 'measured (MEASURED_PEAKS.json)') if 'hbm_gbs' in peaks else (6650.0, 'fallback (B200_PROFILING.md)')
    K = args.steps

    def barrier():
        if dist:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- inputs larger than L2: NB independent copies of the workload (different jitter seeds) stepped round-robin, so every launch finds its
    # state rows in HBM, not in L2
    per_copy = W.footprint(b)
    nb_copies = max(2, -(-int(1.5 * L2_BYTES) // per_copy))
    copies = [b] + [W.make_copy(k) for k in range(1, nb_copies)]
    # untimed set-up: every copy lands and settles under the controller (600 ticks = 0.3 s of simulated time), then W single-tick warm-up launches
    for bk in copies:
        bk.step(600)
    for _ in range(args.warmup):
        for bk in copies:
            bk.step(1)
    torch.cuda.synchronize()
    launches0 = sum(bk.launch_count() for bk in copies)
    sampler = ClockSampler(local_rank) if rank == 0 else None

    def run_block(ticks_per_launch):
        """exactly K steps, bracketed by events on the launching stream; returns (ms, the copy the last launch advanced)"""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        torch.cuda._sleep(2_000_000)   # ~1 ms device-side wait: the first launches queue up behind it, so the window holds no host enqueue gap
        e0.record()
        for i in range(K // ticks_per_launch):
            if ticks_per_launch == 1:
                W.before_step(copies[i % nb_copies], i % nb_copies, nb_copies)
            copies[i % nb_copies].step(ticks_per_launch)
        e1.record()
        barrier()
        return e0.elapsed_time(e1), copies[(K // ticks_per_launch - 1) % nb_copies]

    med, last = run_block(1)                             # headline: single-tick launches
    launches = sum(bk.launch_count() for bk in copies) - launches0
    if args.dump_outputs and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in (('qpos', last.qpos()), ('qvel', last.qvel()), ('time', last.time()), ('obs', last.obs())):
            np.save(os.path.join(args.dump_outputs, name + '.npy'), np.ascontiguousarray(arr, dtype=np.float64))
    T = max(t for t in range(1, 51) if K % t == 0)       # multi-tick launches of T ticks, PD rows held
    med_multi = run_block(T)[0] if T > 1 else med
    # ---- one copy, 256 MiB memset between launches (the other flush method; per-launch events; reported beside the value)
    nfl = min(K, 50)
    evf = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(nfl)]
    for e0, e1 in evf:
        flush.zero_()
        e0.record(); b.step(1); e1.record()
    barrier()
    ms_flush = sum(e0.elapsed_time(e1) for e0, e1 in evf) / nfl
    for bk in copies[1:]:
        bk.close()
    # ---- end to end through the AoS C-ABI: pd_in_t[n] host -> step -> state_out_t[n] host, every step; the whole state_out_t is produced
    # (in-kernel estimator, switched on by the entry point itself).  The estimator-off variant is timed beside it.
    pd = (P.pd_in_t * n)()
    for e in range(n):
        for i in range(5):
            for leg, off in ((pd[e].leftLeg, 0), (pd[e].rightLeg, 5)):
                leg.motorPd.pTarget[i] = PD_TARGET[off + i]; leg.motorPd.pGain[i] = PD_PGAIN[i]; leg.motorPd.dGain[i] = PD_DGAIN[i]
    out = (P.state_out_t * n)()

    def time_e2e():
        for _ in range(4):
            b.L.cassie_sim_step_pd_batch(b.h, C.byref(pd), C.byref(out))
        steps = K
        tm = (C.c_double * 6)()
        b.L.cassie_batch_aos_timing(b.h, tm, 1)
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            b.L.cassie_sim_step_pd_batch(b.h, C.byref(pd), C.byref(out))
        barrier()
        dt = time.perf_counter() - t0
        b.L.cassie_batch_aos_timing(b.h, tm, 1)
        return dt, steps, {'host_pack_ms': 1e3 * tm[0] / max(tm[3], 1), 'device_ms': 1e3 * tm[1] / max(tm[3], 1), 'host_unpack_ms': 1e3 * tm[2] / max(tm[3], 1),
                                'h2d_ms_by_events': tm[4] / max(tm[3], 1) if tm[4] else None, 'kernel_ms_by_events': tm[5] / max(tm[3], 1) if tm[5] else None}
    b.L.cassie_batch_aos_timing.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.c_int]
    t_e2e, e2e_steps, e2e_split = time_e2e()
    full = bool(out[0].pelvis.externalForce[2] != 0 and out[n - 1].leftFoot.toeForce[2] != 0 and out[0].pelvis.position[2] != 0)
    b.enable_estimator_device(False)
    t_e2e_off, e2e_steps_off, _ = time_e2e()
    # the one optional collective of the path (SURVEY 8e): all-gather of every rank's fp32 observation block, timed on its own
    ms_gather = None
    if dist:
        obs_t = b.torch_view('obs')
        gathered = torch.empty((world * n, P.OBS_WIDTH), dtype=torch.float32, device='cuda')
        for _ in range(3):
            dist.all_gather_into_tensor(gathered, obs_t)
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        for _ in range(20):
            dist.all_gather_into_tensor(gathered, obs_t)
        g1.record(); barrier()
        ms_gather = g0.elapsed_time(g1) / 20
    clocks = sampler.stop() if sampler else None
    row_bytes = W.row_bytes(b)
    # ---- the HBM-bound integrate kernel (cassie_batch_integrate_pos) on a state larger than L2
    integ = None
    if rank == 0 and args.config == 2:
        nbi = 1 << 20
        bi = P.CassieBatch(nbi, device=local_rank, precision=P.FP32)
        bi.set_stream(torch.cuda.current_stream().cuda_stream)
        for _ in range(3):
            bi.integrate_pos()
        torch.cuda.synchronize()
        reps = max(10, int(MIN_TIMED_MS / 0.08))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            bi.integrate_pos()
        e1.record(); torch.cuda.synchronize()
        ms_i = e0.elapsed_time(e1) / reps
        bytes_i = nbi * 4 * (35 + 32 + 35)
        integ = {'kernel': 'cassie_integrate_kernel<float>', 'bound': 'hbm', 'achieved': bytes_i / (ms_i * 1e-3) / 1e9, 'peak': hbm_peak, 'unit': 'GB/s',
                 'frac': bytes_i / (ms_i * 1e-3) / 1e9 / hbm_peak, 'traffic': 3.857e8, 'traffic_source': 'static: ncu dram__bytes of profiles/r1_integrate_kernel_ncu_summary.md',
                 'envs': nbi, 'bytes_per_env': 4 * (35 + 32 + 35), 'ms': ms_i, 'launches_timed': reps,
                 'note': 'cassie_integrate_pos (src/cassiemujoco.c:1183-1189): qpos (+)= h qvel, read qpos + qvel, write qpos'}
        bi.close()
    # ---- the other BASELINE configurations beside the headline (short single-tick runs on this GPU; each has its own --config line)
    others = None
    if rank == 0 and args.config == 2 and not args.no_extra:
        others = {}
        for c in (3, 4, 5):
            try:
                Wc = Workload(P, c, CONFIGS[c]['envs'], local_rank, rank, torch)
                bc = Wc.make_copy(0)
                bc.step(600); bc.sync()
                a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                nst = 400 if c == 3 else 120
                a0.record()
                for _ in range(nst):
                    Wc.before_step(bc, 0, 1); bc.step(1)
                a1.record(); torch.cuda.synchronize()
                cn = bc.counters()
                others['config%d' % c] = {'workload': CONFIGS[c]['name'], 'env_steps_per_s': bc.n * nst / (a0.elapsed_time(a1) * 1e-3), 'ms_per_tick': a0.elapsed_time(a1) / nst, 'ticks_timed': nst,
                                          'mean_rows': float(cn[:, 0].mean()), 'mean_pgs_sweeps': float(cn[:, 3].mean()), 'dropped_contacts': int(cn[:, 4].sum()),
                                          'note': 'one copy (L2-warm), single-tick launches; the >L2, >=100 ms figure is bench.py --config %d' % c}
                bc.close()
            except Exception as ex:
                others['config%d' % c] = {'error': repr(ex)}
    # ---- reduce over ranks: a rank's figure is its median block; the job's is the slowest rank's
    t = torch.tensor([med, med_multi, t_e2e / e2e_steps, t_e2e_off / e2e_steps_off, ms_flush], dtype=torch.float64, device='cuda')
    per_rank = None
    if dist:
        allt = torch.empty((world, 5), dtype=torch.float64, device='cuda')
        dist.all_gather_into_tensor(allt, t)
        per_rank = {'kernel_ms_per_step': [float(x) / K for x in allt[:, 0]], 'e2e_ms_per_step': [1e3 * float(x) for x in allt[:, 2]]}
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    med, med_multi, s_e2e, s_e2e_off, ms_flush = [float(x) for x in t]
    if rank == 0:
        try:
            if world > 1 and getattr(args, '_allowed_cpus', None):   # the CPU arm gets the whole lease back (the other ranks are done), not rank 0's pinned share
                os.sched_setaffinity(0, args._allowed_cpus)
            cpu = cpu_baseline(20000 if args.config in (2, 3) else 8000, model=cfg['model'])
        except Exception as ex:   # the oracle is a checker; its absence must not void the GPU number
            cpu = {'value': None, 'unit': 'env-steps/s', 'cores': effective_cpus()[0], 'kind': 'port', 'sample': 'unavailable: %r' % (ex,)}
        ms_step = med / K
        value = world * n / (ms_step * 1e-3)
        ach = row_bytes * n / (ms_step * 1e-3) / 1e9     # algorithmic bytes of one single-tick launch / its duration
        sm_mhz = (clocks or {}).get('sm_mhz') or peaks.get('sm_max_mhz', 1965.0)
        issue_peak = 148 * 4 * sm_mhz * 1e6              # warp instructions / s: 148 SMs x 4 schedulers x clock
        kc = KERNEL_COUNTS.get(str(args.config), {}); inst, inst_src = kc.get('warp_inst_per_env_step'), kc.get('source', 'profiles/r2_step_kernel_counts.json')
        issue = None if inst is None else {'warp_inst_per_env_step': inst, 'source': 'static: ' + inst_src, 'achieved_inst_per_s': inst * value / world, 'peak_inst_per_s': issue_peak,
                                           'frac': inst * value / world / issue_peak, 'sm_mhz': sm_mhz}
        eff = effective_cpus()
        line = {'metric': 'Cassie env-steps/s', 'value': value, 'unit': 'env-steps/s', 'n_gpus': world, 'steps': K, 'warmup': args.warmup,
                'ms_per_step': ms_step, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
                'config': {'workload': cfg['name'], 'envs_per_gpu': n, 'ticks_per_step': 1, 'ticks_per_launch': 1, 'parallelism': 'env-sharded x%d (no data-path collective)' % world,
                           'l2': 'inputs larger than L2: %d independent copies of the batch (%.0f MB) stepped round-robin' % (nb_copies, nb_copies * per_copy / 1e6),
                           'model': 'compiled table of model/%s.xml' % cfg['model']},
                'timing': {'blocks': 1, 'steps_per_block': K, 'timed_ms_total': med,
                           'note': 'exactly K single-tick launches between two CUDA events on the launching stream; max over ranks'},
                'multi_tick_launches': {'ticks_per_launch': T, 'ms_per_step': med_multi / K, 'env_steps_per_s': world * n * K / (med_multi * 1e-3),
                                        'note': 'cassie_batch_step(b, T): T control ticks per launch with the PD rows held, no host round trip; same blocks'},
                'l2_memset_flush_mode': {'ms_per_step': ms_flush, 'env_steps_per_s_this_rank': n / (ms_flush * 1e-3), 'note': 'one copy, 256 MiB memset between launches, per-launch events'},
                'clocks': clocks,
                'e2e': {'value': world * n / s_e2e, 'unit': 'env-steps/s', 'h2d_bytes_per_step': n * P.PD_WIDTH * 4, 'd2h_bytes_per_step': n * P.OBS_WIDTH * 4,
                        'api': 'cassie_sim_step_pd_batch(envs, pd_in_t[n] host, state_out_t[n] host): whole state_out_t incl. the estimator (in-kernel leg-force model + Kalman filters), %d steps, host AoS pack/unpack included' % e2e_steps,
                        'state_out_complete': full, 'split_this_rank_ms': e2e_split, 'host_threads': int(P.lib().cassie_b200_aos_threads()),
                        'estimator_off_variant': {'value': world * n / s_e2e_off, 'note': 'cassie_batch_enable_estimator_device(b, 0): pelvis.position / translationalVelocity / externalForce, terrain.height, toe / heel forces come back zero (partial output)'},
                        'obs_allgather_ms': ms_gather},
                'gpu_launches': launches, 'per_rank': per_rank,
                'roofline': {'kernel': 'cassie_step_kernel<float>', 'bound': 'hbm', 'achieved': ach, 'peak': hbm_peak, 'unit': 'GB/s', 'frac': ach / hbm_peak,
                             'traffic': kc.get('dram_bytes_per_launch'), 'traffic_source': 'static: dram__bytes_read.sum + write.sum of one single-tick launch of this config under ncu --set full (cold caches), ' + str(inst_src),
                             'peak_source': peak_src, 'bytes_per_env_per_launch': row_bytes, 'ticks_per_launch': 1,
                             'issue': issue,
                             'note': 'issue / latency bound by design (SURVEY 8d): the algorithmic HBM traffic is only the persistent state rows in + out, so the HBM fraction is tiny; the issue-slot fraction is the figure that says how far the kernel is from its bound'},
                'roofline_integrate': integ, 'cpu_baseline': cpu, 'other_configs': others}
        print(json.dumps(line, default=lambda o: o.tolist() if hasattr(o, 'tolist') else str(o)), flush=True)
    b.close()
    if dist:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=100)
    ap.add_argument('--warmup', type=int, default=10)
    ap.add_argument('--impl', default='b200')
    ap.add_argument('--config', type=int, default=2, choices=sorted(CONFIGS))
    ap.add_argument('--envs', type=int, default=0, help='environments per GPU (default: the configuration\'s own size)')
    ap.add_argument('--no-extra', dest='no_extra', action='store_true', help='skip the short runs of BASELINE configs 3-5 beside the config-2 line')
    ap.add_argument('--dump-outputs', dest='dump_outputs', metavar='DIR', help='write what the last timed step computed to DIR/<name>.npy')
    args = ap.parse_args()
    rank, local_rank, world = int(os.environ.get('RANK', 0)), int(os.environ.get('LOCAL_RANK', 0)), int(os.environ.get('WORLD_SIZE', 1))
    if args.warmup < 3:
        args.warmup = 3
    if args.steps < 1:
        args.steps = 1
    if args.impl == 'reference':
        reference_arm(args, rank, world)
    else:
        # N ranks on one node share the host: each rank takes its slice of the CPUs (on its GPU's NUMA node) BEFORE any OpenMP runtime starts;
        # the AoS entry point sizes its pack / unpack team from what the process may use
        eff_all, _, quota = effective_cpus()            # before pinning: what the whole job may use
        allowed = sorted(os.sched_getaffinity(0))
        pin_rank_to_its_share(local_rank, world)
        # pack / unpack threads of this rank: its pinned CPUs, but never more than its share of the cgroup quota (N ranks x 32 threads on a lease that
        # owns 64 CPUs would only throttle each other)
        per_rank = max(1, eff_all // max(1, world))
        # ... and two CPUs of the share stay free for the rank's CUDA driver / NCCL / sampler threads: the OpenMP team busy-waits through the whole
        # call, and a job whose teams add up to the quota gets throttled as a whole (8 x 12 threads on a 96-CPU lease: e2e 4 x slower)
        os.environ.setdefault('CASSIE_B200_AOS_THREADS', str(aos_threads_for_rank(effective_cpus()[0], per_rank)))
        args._allowed_cpus = allowed
        gpu_arm(args, rank, local_rank, world)


if __name__ == '__main__':
    main()
