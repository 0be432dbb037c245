#!/usr/bin/env python
"""bench.py -- env-steps/sec of the batched fly environments (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # our CUDA arm
    python bench.py --impl reference --gpus N --steps K ...  # CPU arm: the restated mj_step on the host cores
    python bench.py ... --dump-outputs DIR                   # + the outputs of the last timed step as DIR/*.npy

One "step" = one control step of every environment of the batch (walk: 10 physics substeps of 2e-4 s): workload
`walk_imitation 4096 envs, random policy` per GPU (BASELINE.json configs[1]).  N > 1 is configs[3]: envs sharded across ranks
(weak scaling, 4096 per GPU) and, every control step INSIDE the timed region, the actor-loop exchange over NCCL: actions
[N x 59] scattered from rank 0, task observations (741 floats) + reward + discount + step_type gathered to rank 0.

Steady state (SURVEY.md 8(d) config 2): the env runs with its task hooks on the device (auto-reset at termination / episode end,
observation program, reward); before the warm-up a PRE-ROLL of one episode length (235 control steps) with random actions resets
env e at step hash(e) % 235, so the timed window sees flies at every phase of an episode -- standing, falling, lying on the floor
under random torques -- not the first 50 ms after a standing reset.  `--preroll 0` reproduces the old standing-start window.

  value : env-steps/s, whole job, actions resident in HBM, `env.step_device(actions)` (task hooks + physics + observation
          program, no host copies), device-timed with CUDA events on the stepper's stream, max over ranks; exchange included for N>1
  e2e   : the same metric through the public API `fly_envs.walk_imitation(n_envs, device_task=True).step(host_actions)` with
          pinned host actions in and the observation rows + (reward, discount, step_type) out every step (+ the exchange for N>1)
  extra : (N = 1) the flight_imitation workload (BASELINE.json configs[2]) measured the same way, as a nested block
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ENVS_PER_GPU = 4096
# algorithmic bytes per env-substep (SURVEY.md 8(d)): fp32 state read + written by one physics substep
WORKLOADS = {'walk': dict(model='walk', n_sub=10, bytes_substep=3628, act_scale=0.5, n_action=59, dt='2e-4', episode=235,
                          config='BASELINE.json configs[1]; N>1: configs[3] sharding + NCCL action scatter / observation gather with rank 0'),
             'flight': dict(model='flight', n_sub=4, bytes_substep=1284, act_scale=0.2, n_action=12, dt='5e-5', episode=135,
                            config='BASELINE.json configs[2]: ellipsoid fluid / wing forces, wing-beat pattern generator')}


def measured_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        return json.load(open(p)).get('hbm_gbs', 6650.0), 'measured (MEASURED_PEAKS.json)'
    return 6650.0, 'fallback (B200_PROFILING.md)'


class ClockSampler(threading.Thread):
    def __init__(self, device):
        super().__init__(daemon=True)
        self.device, self.stop_flag, self.samples = device, False, []

    def run(self):
        q = ('index,clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
             'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
        while not self.stop_flag:
            try:
                out = subprocess.run(['nvidia-smi', f'--id={self.device}', f'--query-gpu={q}', '--format=csv,noheader,nounits'],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(',')])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.samples:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        sm = sorted(float(s[1]) for s in self.samples)
        reasons = []
        for i, name in ((3, 'hw_slowdown'), (4, 'hw_thermal_slowdown'), (5, 'sw_thermal_slowdown'), (6, 'sw_power_cap')):
            if any(s[i].lower().startswith('active') for s in self.samples):
                reasons.append(name)
        return {'sm_mhz': sm[len(sm) // 2], 'sm_max_mhz': float(self.samples[0][2]), 'reasons': reasons, 'samples': len(sm)}


DUMP_BUDGET = 64 << 20


def dump_outputs(out_dir, arrays):
    """`--dump-outputs`: the arrays of the last timed step as out_dir/<name>.npy (float32, or float64 for float64 data), so that
    two builds run with the same arguments can be compared output for output.  All arrays share the env axis 0; above
    DUMP_BUDGET bytes a fixed, seeded sample of envs is written instead, and its indices as env_index.npy."""
    arrays = {k: np.asarray(v.detach().cpu().numpy() if hasattr(v, 'detach') else v) for k, v in arrays.items()}
    arrays = {k: v if v.dtype == np.float64 else v.astype(np.float32) for k, v in arrays.items()}
    n = next(iter(arrays.values())).shape[0]
    headers = 128 * (len(arrays) + 1)                                  # .npy headers, env_index.npy included
    if sum(v.nbytes for v in arrays.values()) + headers > DUMP_BUDGET:
        per_env = sum(v.nbytes for v in arrays.values()) // n + 8        # + its float64 entry in env_index
        keep = np.sort(np.random.RandomState(0).choice(n, (DUMP_BUDGET - headers) // per_env, replace=False))
        arrays = {k: v[keep] for k, v in arrays.items()}
        arrays['env_index'] = keep.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, f'{k}.npy'), v)


def start_state(m, wl, rs):
    """the state the CPU arm's single env starts from: the task's reset pose + the bench's joint noise"""
    if wl['model'] == 'flight':
        q = m.qpos0.copy(); q[2] = 1.0
        return q
    q0 = m.qpos0.copy()
    for side in ('left', 'right'):
        for dof, val in (('yaw', 1.5), ('roll', 0.7), ('pitch', -1.0)):
            q0[m.jnt_qposadr_of(f'walker/wing_{dof}_{side}')] = val
    leg = [m.jnt_qposadr[m.actuator_trnid[i]] for i in range(m.nu)
           if m.actuator_trntype[i] == 0 and any(t in m.meta['actuator_names'][i] for t in ('T1', 'T2', 'T3'))]
    q0[leg] += rs.uniform(-0.05, 0.05, len(leg))
    return q0


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_quota():
    """CPU time the container may use, in cores (cgroup v2 cpu.max / v1 cfs quota), or None if unlimited / unknown"""
    try:
        q, p = open('/sys/fs/cgroup/cpu.max').read().split()[:2]
        return None if q == 'max' else float(q) / float(p)
    except Exception:
        pass
    try:
        q = float(open('/sys/fs/cgroup/cpu/cpu.cfs_quota_us').read()); p = float(open('/sys/fs/cgroup/cpu/cpu.cfs_period_us').read())
        return None if q <= 0 else q / p
    except Exception:
        return None


def host_cores():
    """cores this process may run on: the affinity mask, cut to the cgroup's CPU quota (os.cpu_count() is the machine's: a container
    that is allowed 16 cores' worth of time on a 128-core host runs 128 workers at an eighth of their speed each)"""
    try:
        cores = sorted(os.sched_getaffinity(0))
    except AttributeError:
        cores = list(range(os.cpu_count() or 1))
    q = cpu_quota()
    if q is not None and q >= 1 and int(q) < len(cores):
        cores = cores[:int(q)]
    return cores


def cpu_oracle_worker(args):
    """One host core: the restated mj_step (oracle, fp64, MuJoCo's tree-sparse factorisation), one env, random actions, with the
    episode structure of the GPU arm (reset to the start pose every `episode` control steps or on a diverged state)."""
    seed, budget_s, max_steps, core, wl = args
    if core is not None:
        try:
            os.sched_setaffinity(0, {core})
        except Exception:
            pass
    from flybody_b200.flymodel import load_model
    from oracle import fly_oracle as fo
    m = load_model(wl['model'])
    o = fo.Oracle(m)                       # the model's own solver tolerance (1e-8), sparse mode
    rs = np.random.RandomState(seed)
    o.reset(start_state(m, wl, rs))
    acts = rs.uniform(-wl['act_scale'], wl['act_scale'], (256, m.nu))
    phase = int(rs.randint(wl['episode']))         # envs are spread over the phases of an episode, like the GPU arm after its pre-roll
    for k in range(3 + phase % 7):
        o.set(fo.CTRL, acts[k]); o.control_step(wl['n_sub'])
    t0 = time.perf_counter()
    n = 0
    while n < max_steps and time.perf_counter() - t0 < budget_s:
        o.set(fo.CTRL, acts[n % 256]); o.control_step(wl['n_sub'])
        n += 1; phase += 1
        if phase >= wl['episode'] or o.get(fo.FLAGS)[0] != 0:
            o.reset(start_state(m, wl, rs)); phase = 0
    return n, time.perf_counter() - t0


def cpu_baseline(wl, budget_s=10.0, max_steps=100000):
    import multiprocessing as mp
    from oracle import fly_oracle as fo
    fo.build()
    cores = host_cores()
    n1, t1 = cpu_oracle_worker((999, min(2.0, budget_s), max_steps, cores[0], wl))      # one process alone on the box
    with mp.get_context('fork').Pool(len(cores)) as pool:
        res = pool.map(cpu_oracle_worker, [(1000 + i, budget_s, max_steps, c, wl) for i, c in enumerate(cores)])
    rate = sum(n / t for n, t in res)
    return {'value': rate, 'unit': 'env-steps/s', 'cores': len(cores), 'kind': 'port',
            'sample': f'{len(cores)} pinned processes (one per core of os.sched_getaffinity) x ~{budget_s:.0f} s of {wl["model"]}_imitation control steps '
                      f'({wl["n_sub"]} substeps, random actions, reset every {wl["episode"]} steps), oracle/fly_oracle.c: restated mj_step, fp64, '
                      f'gcc -O3 -mavx2, tree-sparse L^T D L + low-rank Newton Hessian as MuJoCo structures it; NOT MuJoCo itself (not installable '
                      f'here); {sum(n for n, _ in res)} env-steps total',
            'per_core': rate / len(cores), 'single_process_per_core': n1 / t1,
            'machine_cpu_count': os.cpu_count(), 'cgroup_cpu_quota_cores': cpu_quota()}


def run_reference(args, wl):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    t0 = time.perf_counter()
    cb = cpu_baseline(wl, budget_s=4.0 * max(1, min(args.steps, 5)))
    wall = time.perf_counter() - t0
    line = {'impl': 'reference', 'metric': f'env-steps/sec on {wl["model"]}_imitation (control steps of {wl["n_sub"]} substeps)', 'value': cb['value'],
            'unit': 'env-steps/s', 'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': 1e3 / cb['per_core'], 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f64', 'data': 'synthetic',
            'config': {'workload': f'{wl["model"]}_imitation, random policy, one env per host core (reference scaling model: '
                                   'one env per actor process, train_dmpo_ray.py:206-227)', 'cores': cb['cores']},
            'cpu_baseline': cb,
            'e2e': {'value': cb['value'], 'unit': 'env-steps/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0, 'wall_s': wall}
    emit(line)


# ------------------------------------------------------------------------------------------------ CUDA arm
def make_env(wl, N, local, seed, device_task=True):
    from flybody_b200 import fly_envs
    if wl['model'] == 'walk':
        return fly_envs.walk_imitation(terminal_com_dist=float('inf'), n_envs=N, device=local, reset_noise=0.05, seed=seed, device_task=device_task)
    return fly_envs.flight_imitation(n_envs=N, device=local, seed=seed, device_task=device_task)


def measure(wl, args, world, rank, local, with_exchange, dump_dir=None):
    """-> dict of raw measurements of one workload on this rank (rank 0 aggregates); with `dump_dir`, the observation rows and
    (reward, discount, step_type) of this rank's envs after the last timed step are written there"""
    import torch
    import torch.distributed as dist
    from flybody_b200 import stepper as st
    dev = torch.device('cuda', local)
    N, K, W, A = args.envs, args.steps, args.warmup, wl['n_action']
    env = make_env(wl, N, local, 1234 + rank, device_task=True)
    env.reset()                                      # SURVEY 8(d) config 2: the INITIAL states carry U(-0.05, 0.05) rad on the leg joints (decorrelation) ...
    if wl['model'] == 'walk':
        env.set_reset_noise(0.0)                     # ... the auto-resets go back to the task's exact start pose, as the reference's do
    sim = env.physics.stepper
    stream = torch.cuda.ExternalStream(sim.stream, device=dev)
    gen = torch.Generator(device=dev); gen.manual_seed(1234 + rank)
    P = args.preroll if args.preroll >= 0 else wl['episode']
    n_act_rows = 64                                                    # a ring of resident random action batches
    acts = (torch.rand((n_act_rows, N, A), device=dev, generator=gen) - 0.5) * (2 * wl['act_scale'])
    # config 4 exchange (flybody_b200.sharding.ActorExchange): rank 0 is the actor (policy side)
    from flybody_b200.sharding import ActorExchange
    xch = ActorExchange(world, rank, N, A, device=dev) if with_exchange else None
    # (a ring of action batches for all ranks: constant actions would drive every fly into its joint limits)
    a_all = (torch.rand((16, world, N, A), device=dev, generator=gen) - 0.5) * (2 * wl['act_scale']) if (with_exchange and rank == 0) else None

    def exchange(obs, out, k):
        """actions for every rank leave rank 0, observations + (reward, discount, step_type) of every rank arrive on rank 0"""
        if not with_exchange:
            return acts[k % n_act_rows]
        if obs is not None:
            xch.gather(obs, out)
        return xch.scatter_actions(a_all[k % 16] if rank == 0 else None)

    state = {'obs': None, 'out': None}

    def one_step(k):
        with torch.cuda.stream(stream):
            a = exchange(state['obs'], state['out'], k)
            state['obs'], state['out'] = env.step_device(a)

    # ---- pre-roll: one episode length with staggered forced resets -> envs at every phase of an episode
    t_pre = time.perf_counter()
    if P > 0:
        ids = np.arange(N)
        slot = ((ids.astype(np.uint64) * np.uint64(2654435761)) >> np.uint64(7)) % np.uint64(P)
        for k in range(P):
            env.request_reset(ids[slot == k])
            one_step(k)
    for k in range(W):
        one_step(k)
    sim.sync(); torch.cuda.synchronize()
    pre_s = time.perf_counter() - t_pre
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local); sampler.start()
    l0 = sim.launch_count
    resets0 = int(env.device_reset_count())
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    with torch.cuda.stream(stream):
        ev0.record(stream)
        for k in range(K):
            one_step(W + k)
        ev1.record(stream)
    sim.sync(); torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1)
    if dump_dir:
        obs, out = state['obs'], state['out']
        dump_outputs(dump_dir, {'observation': obs, 'reward': out[:, 0], 'discount': out[:, 1], 'step_type': out[:, 2]})
    launches = sim.launch_count - l0
    resets = int(env.device_reset_count()) - resets0
    nefc = sim.get(st.NEFC)[:, 0].astype(np.int64); ncon = sim.get(st.NCON)[:, 0].astype(np.int64)
    flags = sim.get(st.FLAGS)[:, 0].astype(np.int64)
    # exchange alone (same buffers, no physics): what the NCCL part costs per control step
    xms = 0.0
    if with_exchange:
        x0, x1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            for k in range(3):
                exchange(state['obs'], state['out'], k)
            x0.record(stream)
            for k in range(K):
                exchange(state['obs'], state['out'], k)
            x1.record(stream)
        torch.cuda.synchronize()
        xms = x0.elapsed_time(x1) / K
    # the same K steps with a CUDA event pair around every kernel launch (cannot replay the step graph -> kept out of `value`)
    sim.profile(True)
    pv0, pv1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        pv0.record(stream)
        for k in range(K):
            one_step(W + K + k)
        pv1.record(stream)
    sim.sync(); torch.cuda.synchronize()
    ms_prof = pv0.elapsed_time(pv1)
    prof = sim.profile_read(); sim.profile(False)
    # ---- e2e through the public API: pinned host actions in, observation rows + (reward, discount, step_type) out, every step
    rs = np.random.RandomState(4321 + rank)
    host_act = torch.empty((K + W, N, A), dtype=torch.float32).pin_memory()
    host_act.copy_(torch.from_numpy(rs.uniform(-wl['act_scale'], wl['act_scale'], (K + W, N, A)).astype(np.float32)))
    a_np = host_act.numpy()
    for k in range(W):
        env.step(a_np[k])
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    t_step = t_x = 0.0
    for k in range(W, W + K):
        ta = time.perf_counter()
        env.step(a_np[k])
        tb = time.perf_counter()
        if with_exchange:
            with torch.cuda.stream(stream):
                exchange(state['obs'], state['out'], k)
        t_step += tb - ta; t_x += time.perf_counter() - tb
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    if os.environ.get('FB_BENCH_DEBUG'):
        print(f'[rank {rank}] e2e loop: env.step {t_step / K * 1e3:.2f} ms, exchange enqueue {t_x / K * 1e3:.2f} ms, total {e2e_s / K * 1e3:.2f} ms per step', file=sys.stderr, flush=True)
    sampler.stop_flag = True; sampler.join(timeout=2)
    if world > 1:
        t = torch.tensor([ms, e2e_s, xms], device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX); ms, e2e_s, xms = [float(x) for x in t.tolist()]
        r = torch.tensor([resets, int((flags & 1).sum()), int(((flags & 6) != 0).sum())], device=dev); dist.all_reduce(r); resets, bad, over = [int(x) for x in r.tolist()]
    else:
        bad, over = int((flags & 1).sum()), int(((flags & 6) != 0).sum())
    res = dict(ms=ms, e2e_s=e2e_s, xms=xms, launches=int(launches), prof=prof, ms_prof=ms_prof, resets=resets, bad=bad, over=over, pre_s=pre_s, P=P,
               clocks=sampler.summary(), h2d=int(env.h2d_bytes_per_step), d2h=int(env.d2h_bytes_per_step), record_bytes=int(sim.record_bytes),
               obs_dim=int(state['obs'].shape[1]),
               nefc_hist={f'<={b}': int((nefc <= b).sum()) for b in (8, 16, 24, 32, 48, 64, 96, 128, 160)}, nefc_mean=float(nefc.mean()), nefc_max=int(nefc.max()),
               ncon_mean=float(ncon.mean()), ncon_max=int(ncon.max()), share_global_solver=float((nefc > 32).mean()))
    env.close()
    return res


def line_of(wl, args, world, r):
    N, K = args.envs, args.steps
    peak, peak_src = measured_peaks()
    total = N * world
    prof = r['prof']
    stage = {k: v for k, v in prof.items() if v[1] > 0}
    dom_name, (dom_ms, dom_n) = max(stage.items(), key=lambda kv: kv[1][0])
    step_ms_sum = sum(v[0] for v in stage.values())
    avg_launch_s = dom_ms / max(dom_n, 1) * 1e-3
    substeps_per_launch = max(1, round(K * wl['n_sub'] / max(dom_n, 1)))
    achieved = wl['bytes_substep'] * N * substeps_per_launch / avg_launch_s / 1e9
    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, 'profiles', 'dominant_kernel_traffic.json')
    if os.path.exists(tp):
        t = json.load(open(tp))
        ent = t.get('kernels', {}).get(f'{wl["model"]}:{dom_name}')
        if ent:
            traffic, traffic_src = ent['dram_bytes_per_launch'], ent.get('source')
    bytes_step = wl['bytes_substep'] * wl['n_sub']
    return {
        'metric': f'env-steps/sec on {wl["model"]}_imitation (control steps of {wl["n_sub"]} substeps)', 'value': total * K / (r['ms'] * 1e-3), 'unit': 'env-steps/s',
        'n_gpus': world, 'steps': K, 'warmup': args.warmup, 'ms_per_step': r['ms'] / K, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': f'{wl["model"]}_imitation {N} envs per GPU, random policy U(-{wl["act_scale"]},{wl["act_scale"]}), {wl["n_sub"]} substeps x {wl["dt"]} s ({wl["config"]})',
                   'envs_per_gpu': N, 'total_envs': total, 'n_substeps': wl['n_sub'],
                   'steady_state': f'pre-roll of {r["P"]} control steps with staggered forced resets (envs at every phase of a {wl["episode"]}-step episode), then {args.warmup} warm-up steps; '
                                   f'{r["resets"]} auto-resets inside the timed window (counted in the work)' if r['P'] > 0 else 'no pre-roll: standing start',
                   'constraint_rows': {'mean': r['nefc_mean'], 'max': r['nefc_max'], 'hist_envs': r['nefc_hist'], 'contacts_mean': r['ncon_mean'], 'contacts_max': r['ncon_max'],
                                       'share_of_envs_on_global_memory_solver_path(nefc>32)': r['share_global_solver']},
                   'l2': f'inputs larger than L2: every launch streams the env records ({r["record_bytes"] / 1e3:.0f} KB each, {r["record_bytes"] * N / 1e9:.2f} GB per GPU vs 126 MB L2); no explicit flush',
                   'parallelism': f'env-sharded x{world}' + (f', per control step inside the timed region: NCCL scatter of actions [{total}x{wl["n_action"]}] from rank 0 + gather of task observations '
                                                             f'[{total}x{r["obs_dim"]}] and (reward, discount, step_type) to rank 0; exchange alone {r["xms"]:.3f} ms/step '
                                                             f'({100 * r["xms"] / (r["ms"] / K):.1f} % of the step), limiter: rank-0 NVLink ingest of the gather' if world > 1 else ''),
                   'diverged_envs_flagged': r['bad'], 'capacity_overflow_envs_flagged': r['over'], 'preroll_wall_s': r['pre_s']},
        'clocks': r['clocks'], 'gpu_launches': r['launches'],
        'e2e': {'value': total * K / r['e2e_s'], 'unit': 'env-steps/s', 'h2d_bytes_per_step': r['h2d'], 'd2h_bytes_per_step': r['d2h'],
                'api': f'flybody_b200.fly_envs.{wl["model"]}_imitation(n_envs, device_task=True).step(action)' + (' on every rank + the rank-0 exchange' if world > 1 else '')},
        'roofline': {'bound': 'hbm', 'kernel': dom_name, 'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak,
                     'traffic': traffic, 'traffic_source': traffic_src, 'peak_source': peak_src,
                     'how': f'algorithmic bytes = {wl["bytes_substep"]} B/env-substep x {N} envs x {substeps_per_launch} substep(s) per launch / mean CUDA-event duration of the '
                            f'"{dom_name}" kernel over a second pass of the same {K} steps with an event pair around every launch ({dom_n} launches, '
                            f'{r["ms_prof"] / K:.3f} ms per step in that pass; `value` is the pass without per-launch events, which replays the step graph); whole-step algorithmic GB/s = '
                            f'{bytes_step * total * K / (r["ms"] * 1e-3) / 1e9:.2f}',
                     'kernel_share': dom_ms / max(step_ms_sum, 1e-9),
                     'stage_ms_per_step': {k: v[0] / K for k, v in stage.items()}},
    }


def measure_vision(args, world, rank, local, n_envs=1024, dump_dir=None):
    """BASELINE.json configs[4] shape: `vision_guided_flight` (heightfield terrain contacts, two 32 x 32 x 3 eye cameras rendered on the
    device every step, wing-beat pattern generator, the task's hooks as device code: fb_task_* kind 2) + the reference's vision policy
    (VisNet + two-level controller, flybody_b200/policy_torch.py, random weights) in the loop on rank 0 (observation rows + eyes of all
    ranks gathered over NCCL, actions scattered back).  `value`: everything stays in HBM (`step_device`: torch views of the rows and the
    eye images).  `e2e`: env.step(host actions) -> observations + eyes on the host -> policy input copied up -> actions copied down.
    With `dump_dir`: the rows, (reward, discount, step_type), eyes and policy actions of this rank after the last timed step."""
    import torch
    import torch.distributed as dist
    from flybody_b200 import fly_envs
    from flybody_b200.policy_torch import vision_policy_for
    dev = torch.device('cuda', local)
    K, W, N = args.steps, args.warmup, n_envs
    env = fly_envs.vision_guided_flight(n_envs=N, device=local, seed=1234 + rank, terrain_bank=64, device_task=True)
    ts = env.reset()
    vis, ctl, keys = vision_policy_for(env, device=dev)
    spec = env.action_spec()
    lo, hi = torch.tensor(spec.minimum, device=dev, dtype=torch.float32), torch.tensor(spec.maximum, device=dev, dtype=torch.float32)
    A = spec.shape[0]
    layout = env.observation_layout()
    keys = [k for k in keys if k in layout and layout[k].stop > layout[k].start]          # (actuator_activation is empty for this model)
    col_task = torch.arange(layout['walker/task_input'].start, layout['walker/task_input'].stop, device=dev)
    col_others = torch.cat([torch.arange(layout[k].start, layout[k].stop, device=dev) for k in keys])
    bufs = {}

    def policy(eyes, task, others):
        left, right = eyes[:, 1], eyes[:, 0]
        if world > 1:
            if not bufs:
                for name, t in (('left', left), ('right', right), ('task', task), ('others', others)):
                    bufs[name] = [torch.empty_like(t) for _ in range(world)] if rank == 0 else None
                bufs['a_loc'] = torch.empty((N, A), device=dev)
            for name, t in (('left', left), ('right', right), ('task', task), ('others', others)):
                dist.gather(t.contiguous(), bufs[name], dst=0)
            if rank == 0:
                left, right, task, others = (torch.cat(bufs[n]) for n in ('left', 'right', 'task', 'others'))
        a = None
        if rank == 0:
            with torch.no_grad():
                a = torch.minimum(torch.maximum(ctl(vis(left, right, task, others)), lo), hi)
        if world > 1:
            dist.scatter(bufs['a_loc'], [a[r * N:(r + 1) * N].contiguous() for r in range(world)] if rank == 0 else None, src=0)
            a = bufs['a_loc']
        return a.contiguous()

    def act_host(ts):                                       # observations on the host (the dm_env contract) -> policy input copied up
        o = ts.observation
        eyes = torch.from_numpy(np.stack([np.asarray(o['walker/right_eye']), np.asarray(o['walker/left_eye'])], 1)).to(dev)
        task = torch.from_numpy(np.asarray(o['walker/task_input'], np.float32)).to(dev)
        others = torch.from_numpy(np.concatenate([np.asarray(o[k], np.float32).reshape(N, -1) for k in keys], 1)).to(dev)
        return policy(eyes, task, others).cpu().numpy()

    def act_dev(rows, eyes):
        return policy(eyes, rows[:, col_task], rows[:, col_others])

    def sync():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def maxr(x):
        if world > 1:
            t = torch.tensor([x], device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX); return float(t.item())
        return x

    # ---- device-resident arm: the policy runs on the stepper's stream, ordered after the step and the eye render
    stream = torch.cuda.ExternalStream(env._sim.stream, device=dev)
    with torch.cuda.stream(stream):
        a = torch.zeros((N, A), device=dev)
        for k in range(max(W, 3)):
            rows, out, eyes = env.step_device(a)
            a = act_dev(rows, eyes)
        sync()
        l0 = env._sim.launch_count
        e0 = env._sim.task_episodes().sum()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        for k in range(K):
            rows, out, eyes = env.step_device(a)
            a = act_dev(rows, eyes)
        ev1.record(stream)
        sync()
        if dump_dir:
            dump_outputs(dump_dir, {'observation': rows, 'reward': out[:, 0], 'discount': out[:, 1], 'step_type': out[:, 2], 'eyes': eyes, 'action': a})
        dt_dev = maxr(ev0.elapsed_time(ev1) * 1e-3)
        launches = env._sim.launch_count - l0
        resets = int(env._sim.task_episodes().sum() - e0)
        env._sim.profile(True)
        for k in range(5):
            rows, out, eyes = env.step_device(a)
            a = act_dev(rows, eyes)
        torch.cuda.synchronize()
    prof = {k: v[0] / 5 for k, v in env._sim.profile_read().items() if v[1]}
    env._sim.profile(False)
    # ---- end-to-end arm (host observations, host actions)
    ts = env.reset()
    for k in range(max(W, 3)):
        ts = env.step(act_host(ts))
    sync()
    t0 = time.perf_counter()
    for k in range(K):
        ts = env.step(act_host(ts))
    sync()
    dt = maxr(time.perf_counter() - t0)
    eyes_bytes = int(np.asarray(ts.observation['walker/left_eye']).nbytes * 2)
    obs_bytes = int(env._rec.nbytes + env._out4.nbytes)
    pol_bytes = int(sum(np.asarray(ts.observation[k]).reshape(N, -1).shape[1] for k in keys) * N * 4 + N * 2 * 4)
    total = N * world
    res = {'metric': 'env-steps/sec on vision_guided_flight + vision policy in the loop (control steps of 4 substeps)', 'value': total * K / dt_dev, 'unit': 'env-steps/s',
           'ms_per_step': dt_dev / K * 1e3, 'n_gpus': world, 'gpu_launches': int(launches),
           'config': {'workload': f'vision_guided_flight {N} envs per GPU (BASELINE.json configs[4]: 1024 per GPU), bumps terrain 401 x 401 per env from a device bank of 64, '
                                  'task hooks on the device (fb_task_* kind 2), eyes 2 x 32 x 32 x 3 uint8 rendered every step, '
                                  'policy = VisNet + TwoLevelController (torch, random weights) on rank 0',
                      'envs_per_gpu': N, 'total_envs': total, 'auto_resets_in_window': resets,
                      'note': '`value`: observation rows, eyes and actions stay in HBM (step_device); `e2e`: the dm_env-style env.step() with host buffers'},
           'e2e': {'value': total * K / dt, 'unit': 'env-steps/s', 'ms_per_step': dt / K * 1e3,
                   'h2d_bytes_per_step': int(N * A * 4 + eyes_bytes + pol_bytes), 'd2h_bytes_per_step': int(eyes_bytes + obs_bytes + N * A * 4),
                   'api': 'flybody_b200.fly_envs.vision_guided_flight(n_envs, device_task=True).step(action) + policy_torch.VisNet / TwoLevelController'},
           'stage_ms_per_step': prof}
    env.close()
    return res


def run_ours(args, wl):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device; the stepper has no CPU path (use --impl reference for the CPU arm)')
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault('NCCL_DEBUG_FILE', '/dev/stderr')      # stdout carries exactly one JSON line
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    if args.workload == 'vision':
        res = measure_vision(args, world, rank, local, n_envs=args.envs if args.envs != ENVS_PER_GPU else 1024,
                             dump_dir=args.dump_outputs if rank == 0 else None)
        if rank == 0:
            res.update({'steps': args.steps, 'warmup': args.warmup, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic'})
            emit(res)
        if world > 1:
            dist.barrier(); dist.destroy_process_group()
        return
    r = measure(wl, args, world, rank, local, with_exchange=world > 1, dump_dir=args.dump_outputs if rank == 0 else None)
    if rank == 0:
        line = line_of(wl, args, world, r)
        if world == 1 and not args.no_extra and args.workload == 'walk':
            wf = WORKLOADS['flight']
            try:
                rf = measure(wf, args, 1, 0, local, False)
                lf = line_of(wf, args, 1, rf)
                line['extra'] = {'flight_imitation': {k: lf[k] for k in ('metric', 'value', 'unit', 'ms_per_step', 'config', 'gpu_launches', 'e2e', 'roofline')}}
            except Exception as e:                                   # the headline must not depend on the extra block
                line['extra'] = {'flight_imitation': {'error': repr(e)}}
            try:
                line['extra']['vision_guided_flight'] = measure_vision(args, 1, 0, local)
            except Exception as e:
                line['extra']['vision_guided_flight'] = {'error': repr(e)}
        if world == 1 and not args.no_cpu:
            line['cpu_baseline'] = cpu_baseline(wl, budget_s=args.cpu_seconds)
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


_JSON_FD = None


def emit(line):
    """the one JSON line of this run, on the process's ORIGINAL stdout (see main)"""
    data = (json.dumps(line) + '\n').encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def main():
    # stdout carries exactly one JSON line: everything else that writes to fd 1 (the NCCL version banner, library chatter of the
    # worker processes) is sent to stderr for the whole run
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--envs', type=int, default=ENVS_PER_GPU, help='envs per GPU')
    ap.add_argument('--cpu-seconds', type=float, default=10.0)
    ap.add_argument('--no-cpu', action='store_true')
    ap.add_argument('--no-extra', action='store_true', help='skip the nested flight_imitation block')
    ap.add_argument('--preroll', type=int, default=-1, help='control steps of staggered-reset pre-roll before the warm-up (-1: one episode length; 0: standing start)')
    ap.add_argument('--workload', default='walk', choices=sorted(WORKLOADS) + ['vision'], help='walk = the headline (BASELINE configs[1]); flight = configs[2]')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help="CUDA arm: write what the timed path returned in its last step (rank 0's envs) as DIR/<name>.npy, at most 64 MB; "
                         'the inputs are seeded, so runs with the same arguments can be compared output for output')
    args = ap.parse_args()
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs covers the CUDA arm only: the reference arm runs for a time budget, not a number of steps')
    args.warmup = max(args.warmup, 3)
    wl = WORKLOADS.get(args.workload, WORKLOADS['flight'])
    if args.impl == 'reference':
        run_reference(args, wl)
    else:
        run_ours(args, wl)


if __name__ == '__main__':
    main()
