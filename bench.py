#!/usr/bin/env python
"""Benchmark of the local-energy hot path (contract in the task statement / DESIGN.md).

  python bench.py --gpus N --steps K --warmup W            # our arm (CUDA engine)
  python bench.py --impl reference --steps K --warmup W    # reference arm: CPU oracle port
  python bench.py ... --dump-outputs DIR                   # also write the last timed step's outputs as DIR/<name>.npy

metric: walker.local-energies / second.  A "step" = one local-energy evaluation of every walker
of the batch (Psiformer forward + forward-Laplacian + potentials, incl. the non-local ECP
quadrature) followed, for N > 1, by the fused statistics all-reduce.  Default workload = the
configuration BASELINE.json's metric is quoted on: benzene (ccECP, 30 valence electrons)
Psiformer (d=256, L=4, H=4, K=16), a GLOBAL batch of 4096 walkers split over the N GPUs as the
reference splits electron_batch_size over its devices (parallel.py:296-317; "scaling": "strong";
``--scaling weak`` keeps 4096 walkers per GPU instead).  The engine chunks the walkers through its
workspace, so the whole batch fits one B200.  ``--workload lih_psiformer`` = BASELINE configs[1],
``n2_ferminet`` = configs[2].  Synthetic walkers (atom-centred Gaussians, equilibrated by
Metropolis sub-steps, untimed) and random-init weights.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np
import torch

WORKLOADS = {
    'lih_psiformer': dict(mol='LiH', ecp=None, walkers=4096, hyper={}, kind='psiformer'),
    'n2_psiformer': dict(mol='N2', ecp=None, walkers=4096, hyper={}, kind='psiformer'),
    'n2_ferminet': dict(mol='N2', ecp=None, walkers=4096, hyper={}, kind='ferminet'),
    'benzene_psiformer': dict(mol='benzene', ecp='ccECP', walkers=4096, hyper={}, kind='psiformer'),
    'lih_paulinet': dict(mol='LiH', ecp=None, walkers=256, hyper={}, kind='paulinet'),  # BASELINE configs[0]
    # the one step rate the reference publishes for this path (BASELINE.md 1): evaluation of the LiH Psiformer with 2048
    # walkers, a step = DecorrSampler(30) Metropolis sub-steps + E_loc, 2.16 it/s on an RTX 3090
    # (doc/examples/ground_state_lih.ipynb:227,238; sampling/electron_samplers.py:347-357)
    'lih_eval_step': dict(mol='LiH', ecp=None, walkers=2048, hyper={}, kind='psiformer', mcmc_substeps=30,
                          published_it_per_s=2.16),
    # BASELINE configs[4]: excited-state penalty run, 2 electronic states, 2048 walkers per state
    # (conf/task/train_excited_psiformer.yaml:25, conf/ansatz/transpsiformer.yaml, conf/hamil/mol/cyclobutadiene_square.yaml)
    'cyclobutadiene_transpsiformer': dict(mol='cyclobutadiene_square', ecp=None, walkers=2048, hyper={}, kind='transpsiformer',
                                          states=2),
}


def algorithmic_flops_per_eloc(N, M, d=256, L=4, K=16, n_ecp=0):
    """SURVEY.md 8(d): F_lap with dense 3N tangents (forward-Laplacian) + 12 N N_ecp plain forwards."""
    T = 3 * N
    f_lap = (5 * 2 * N * (4 * M + 1) * d + (T + 2) * (L * 12 * N * d * d + 2 * K * N * N * d + 6 * K * N * N * M)
             + (3 * T + 3) * L * 4 * N * N * d + K * (2 / 3 + 2) * N**3 + 2 * K * T * N**3)
    f_fwd = 2 * N * (4 * M + 1) * d + L * (12 * N * d * d + 4 * N * N * d) + 2 * K * N * N * d + 6 * K * N * N * M + 2 / 3 * K * N**3
    return f_lap + 12 * N * n_ecp * f_fwd


def make_problem(wl, B, seed):
    from deepqmc_b200 import params as PN
    from deepqmc_b200.hamil import MolecularHamiltonian
    from deepqmc_b200.molecule import Molecule

    mol = Molecule.from_name(wl['mol'])
    hamil = MolecularHamiltonian(mol=mol, ecp_type=wl['ecp'])
    rng = np.random.default_rng(seed)
    N = hamil.n_up + hamil.n_down
    p = hamil.ns_valence / hamil.ns_valence.sum()
    centers = rng.choice(len(mol.coords), size=(B, N), p=p)
    r = mol.coords[centers] + rng.normal(size=(B, N, 3)) * 0.7
    return mol, hamil, r, PN


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    Q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--id={self.index}', f'--query-gpu={self.Q}',
                                          '--format=csv,noheader,nounits', '-lms', '100'], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(',')])

    def stop(self):
        if not self.proc:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace('.', '').isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace('.', '').isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = sorted({n for r in self.rows if len(r) >= 6 for n, v in zip(names, r[2:6]) if v.lower().startswith('active')})
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': reasons, 'samples': len(sm)}


# dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel from one
# `ncu --set full` capture of the same command (profiles/, B200_PROFILING.md); None = not captured.
TRAFFIC = {
    # profiles/r02_ncu_trunk_f16_kernel_ts.csv (ncu --set full of `tools/prof_fwd.py 2 17760`): one whole-trunk launch over
    # 17760 plain-forward walkers x 30 electrons = 532800 rows: dram read 0.705 GB + write 2.368 GB.  Algorithmic bytes of
    # that launch = rows x 256 x 4 B in + the same out + 6.3 MB of weights = 1.097 GB: the extra ~1.8 GB of writes are
    # evictions of the per-CTA Q/K/V operand scratch (57 MB, re-written every tile and layer) from L2.  (The quadrature
    # forwards of the ECP pass read even less: the unmoved electrons' embedding rows come from the base walkers' table.)
    'benzene_psiformer': {'bytes_per_launch': 3.0727e9, 'algorithmic_bytes_per_launch': 1.0975e9,
                          'launch': 'trunk_f16_kernel<TS>, 532800 rows (17760 plain-forward walkers x 30 electrons), 4 layers',
                          'source': 'profiles/r02_ncu_trunk_f16_kernel_ts.csv'},
}

DUMP_LIMIT_BYTES = 64 * 1024 * 1024


def dump_outputs(out_dir, per_walker, other):
    """Write one step's outputs as ``out_dir/<name>.npy`` in float32 or float64, so that two builds run with the same
    arguments can be compared array by array.  ``per_walker`` arrays share a leading walker axis; if everything together
    would exceed 64 MiB, they are cut to a fixed, seeded sample of walkers and ``walker_index.npy`` names the walkers kept."""
    def host(x):
        x = x.detach().cpu().numpy() if torch.is_tensor(x) else np.asarray(x)
        return x.astype(np.float64 if x.dtype == np.float64 else np.float32)

    per_walker = {k: host(v) for k, v in per_walker.items()}
    other = {k: host(v) for k, v in other.items()}
    n = next(iter(per_walker.values())).shape[0]
    walker_bytes = sum(v.nbytes for v in per_walker.values()) // n
    budget = DUMP_LIMIT_BYTES - sum(v.nbytes for v in other.values())
    if walker_bytes * n > budget:
        keep = budget // (walker_bytes + 8)  # 8 bytes per walker for walker_index itself
        idx = np.sort(np.random.default_rng(0).choice(n, size=keep, replace=False))
        per_walker = {k: v[idx] for k, v in per_walker.items()}
        other['walker_index'] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in {**per_walker, **other}.items():
        np.save(os.path.join(out_dir, f'{k}.npy'), v)


_ORACLE = {}


def _oracle_init(wl_name, seed):
    """Pool initialiser: one single-threaded oracle per worker process."""
    torch.set_num_threads(1)
    from deepqmc_b200.spec import ferminet_spec, paulinet_spec, psiformer_spec, transpsiformer_spec
    from oracle import wf
    from oracle.hamil import OracleHamiltonian

    wl = WORKLOADS[wl_name]
    mol, hamil, r, PN = make_problem(wl, 1, seed)
    oh = OracleHamiltonian(mol, ecp_type=wl['ecp'])
    spec = {'psiformer': psiformer_spec, 'ferminet': ferminet_spec, 'paulinet': paulinet_spec,
            'transpsiformer': transpsiformer_spec}[wl['kind']](oh, **wl['hyper'])
    pt = wf.to_torch(PN.perturb_params(PN.init_params(spec, 0)))
    J = 0 if oh.nl_params is None else len(np.unique(np.nonzero(oh.nl_params)[0]))
    _ORACLE.update(wl=wl, oh=oh, spec=spec, pt=pt, R=torch.as_tensor(mol.coords), J=J, wf=wf)


def _oracle_eval(r_np):
    o = _ORACLE
    f = lambda x: o['wf'].log_psi(o['spec'], o['pt'], x, o['R'])
    tw = torch.zeros(max(o['J'], 1), o['spec'].n_elec) + 0.1
    e, _ = o['oh'].local_energy(f, torch.as_tensor(r_np), o['R'], phi_random=tw if o['J'] else None)
    return float(e)


def _oracle_task(task):
    """One slice of ONE walker's local energy (heavy workloads: a single benzene walker costs about
    a minute of one core, so its 3N Hessian rows and its 12 N N_ecp quadrature forwards are spread
    over the worker processes).  kind 'lap': Hessian rows [lo, hi) (+ gradient and the local
    potentials with the first slice); kind 'ecp': (nucleus, electron) pairs [lo, hi)."""
    r_np, kind, lo, hi = task
    o = _ORACLE
    r = torch.as_tensor(r_np)
    f = lambda x: o['wf'].log_psi(o['spec'], o['pt'], x, o['R'])
    if kind == 'lap':
        x = r.reshape(-1)
        grad_f = torch.func.grad(lambda xx: f(xx.reshape(-1, 3))[1])
        eye = torch.eye(x.numel(), dtype=x.dtype)[lo:hi]
        rows = torch.func.vmap(lambda v: torch.func.jvp(grad_f, (x,), (v,))[1])(eye)
        out = float(rows[torch.arange(hi - lo), torch.arange(lo, hi)].sum())
        if lo == 0:  # E_loc = -(lap + |g|^2)/2 + potentials (oracle/hamil.py local_energy)
            g = grad_f(x)
            oh = o['oh']
            out = -0.5 * (out + float((g * g).sum())) + float(oh.nuclear_energy(o['R']) + oh.electronic_potential(r)
                                                               + oh.local_potential(r, o['R']))
        else:
            out = -0.5 * out
        return out
    tw = torch.zeros(max(o['J'], 1), o['spec'].n_elec) + 0.1
    N = o['spec'].n_elec
    pairs = {(p // N, p % N) for p in range(lo, hi)}
    return float(o['oh'].nonloc_potential(r, o['R'], f, tw, pairs=pairs))


def time_oracle(wl_name, per_worker, steps, warmup, seed=0):
    """CPU arm: the oracle (torch fp64 restatement of the reference path) on the host cores, one
    single-threaded process per core.  Light workloads: whole walkers per worker (the walker axis
    is embarrassingly parallel, which is also how XLA:CPU would spread the reference's vmap).
    Heavy workloads (non-local ECP): a step is a bounded sample of `per_worker` walkers whose
    Hessian rows / quadrature pairs are spread over all workers.  Returns walkers/s, workers,
    ms/step, walkers per step."""
    import multiprocessing as mp

    workers = max(1, len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1))
    wl = WORKLOADS[wl_name]
    heavy = wl['ecp'] is not None
    n = per_worker if heavy else workers * per_worker
    _, hamil, r, _ = make_problem(wl, n * (steps + warmup), seed)
    times = []
    with mp.get_context('fork').Pool(workers, initializer=_oracle_init, initargs=(wl_name, seed)) as pool:
        if heavy:
            N = hamil.n_up + hamil.n_down
            n_pairs = N * len(hamil.pot.nuc_with_nl_pot)

            def tasks(rw):
                t = [(rw, 'lap', lo, min(lo + 6, 3 * N)) for lo in range(0, 3 * N, 6)]
                return t + [(rw, 'ecp', lo, min(lo + 2, n_pairs)) for lo in range(0, n_pairs, 2)]

            pool.map(_oracle_task, [(r[0], 'ecp', i % n_pairs, i % n_pairs + 1) for i in range(workers)])  # first-call cost
            for s in range(steps + warmup):
                t0 = time.perf_counter()
                todo = [t for i in range(n) for t in tasks(r[s * n + i])]
                pool.map(_oracle_task, todo, chunksize=1)
                dt = time.perf_counter() - t0
                if s >= warmup:
                    times.append(dt)
        else:
            pool.map(_oracle_eval, [r[i] for i in range(workers)])  # import / first-call cost, untimed
            for s in range(steps + warmup):
                t0 = time.perf_counter()
                pool.map(_oracle_eval, [r[s * n + i] for i in range(n)], chunksize=per_worker)
                dt = time.perf_counter() - t0
                if s >= warmup:
                    times.append(dt)
    return n * len(times) / sum(times), workers, 1e3 * float(np.mean(times)), n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='benzene_psiformer', choices=sorted(WORKLOADS))
    ap.add_argument('--dtype', default='float32', choices=['float32', 'float64'])
    ap.add_argument('--walkers', type=int, default=None, help='walker batch: global (strong scaling) or per GPU (weak)')
    ap.add_argument('--scaling', default='strong', choices=['strong', 'weak'],
                    help='strong (default): the global batch is split over the GPUs as the reference does; weak: per-GPU batch')
    ap.add_argument('--cpu-sample', type=int, default=None)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--gemm-backend', default='tcgen05', choices=['simt', 'tcgen05'])
    ap.add_argument('--equil-sweeps', type=int, default=None)
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help="write what the last timed step computed (rank 0's walkers) as DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error('--steps must be at least 1')
    if a.dump_outputs and a.impl == 'reference':
        ap.error('--dump-outputs writes the outputs of the CUDA engine; the reference arm keeps none')
    wl = WORKLOADS[a.workload]
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    B_global = (a.walkers or wl['walkers']) * (world if a.scaling == 'weak' else 1)
    if B_global % world:
        raise SystemExit('the walker batch must be divisible by the number of GPUs (reference validate_kwargs.py:45-48)')
    B = B_global // world  # walkers of this rank
    unit = 'walker.local-energies/s'
    metric = 'walker.local-energies/sec'
    arch = {'psiformer': 'Psiformer d256 L4 H4 K16', 'ferminet': 'FermiNet d256 L4 e32 K16',
            'transpsiformer': 'TransPsiformer d256 L4 H4 K16',
            'paulinet': 'PauliNet test ansatz (tests/conf/ansatz.yaml) d8 L1 K2'}[wl['kind']]
    n_states = wl.get('states', 1)
    workload_name = f"{wl['mol']} {arch}{' ' + wl['ecp'] if wl['ecp'] else ''}, {B_global} walkers" + (
        f' per state x {n_states} electronic states (energies + pairwise overlap penalty)' if n_states > 1 else '')

    if a.impl == 'reference':
        if rank != 0:
            return 0
        heavy = wl['ecp'] is not None
        per_worker = a.cpu_sample or (8 if wl['mol'] == 'LiH' else (2 if heavy else 1))
        val, cores, ms, n_sample = time_oracle(a.workload, per_worker, a.steps, a.warmup)
        how = ('Hessian rows and ECP quadrature pairs of each walker spread over one single-threaded process per core'
               if heavy else 'one single-threaded process per core')
        out = {
            'impl': 'reference', 'metric': metric, 'value': val, 'unit': unit, 'n_gpus': a.gpus, 'steps': a.steps,
            'warmup': a.warmup, 'ms_per_step': ms, 'higher_is_better': True, 'scaling': a.scaling, 'vs_baseline': None,
            'dtype': 'f64', 'data': 'synthetic',
            'config': {'workload': workload_name, 'note': 'CPU oracle port of the reference JAX path (JAX not installable here)'},
            'cpu_baseline': {'value': val, 'unit': unit, 'cores': cores, 'kind': 'port',
                             'sample': f'{n_sample} walkers per step x {a.steps} steps, {how} (autograd-Hessian Laplacian, fp64)'},
            'e2e': {'value': val, 'unit': unit, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        }
        print(json.dumps(out))
        return 0

    # ------------------------------- our arm -------------------------------------------------
    from deepqmc_b200 import parallel
    from deepqmc_b200.ansatz import B200Ansatz
    from deepqmc_b200.types import PhysicalConfiguration

    assert torch.cuda.is_available(), 'bench.py needs a CUDA device; there is no CPU fallback (use --impl reference)'
    if world > 1:  # communicator set-up is logged (rank count, transport) so that the run shows which collective path it used
        os.environ.setdefault('NCCL_DEBUG', 'INFO')
        os.environ.setdefault('NCCL_DEBUG_SUBSYS', 'INIT')
    rank, world = parallel.init_from_env()
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    mol, hamil, r_np, PN = make_problem(wl, B_global * n_states, seed=1000)
    r_np = r_np.reshape(n_states, B_global, *r_np.shape[1:])[:, rank * B:(rank + 1) * B]  # contiguous walker block of this rank
    backend = 1 if (a.gemm_backend == 'tcgen05' and a.dtype == 'float32' and wl['kind'] != 'paulinet') else 0  # d = 8: CUDA cores
    ansatz = B200Ansatz(hamil, wl['kind'], dtype=a.dtype, device=local, gemm_backend=backend, **wl['hyper'])
    # one parameter tree per electronic state (excited-state runs: reference wf/base.py:27-44 stacks them on a state axis)
    params_all = [PN.perturb_params(ansatz.init(st), seed=st) for st in range(n_states)]
    params = params_all[0]
    tdt = torch.float32 if a.dtype == 'float32' else torch.float64
    N, M = hamil.n_up + hamil.n_down, hamil.n_nuc
    n_ecp = len(hamil.pot.nuc_with_nl_pot)
    R = torch.as_tensor(mol.coords, dtype=tdt, device=dev)
    heavy = wl['ecp'] is not None
    n_equil = a.equil_sweeps if a.equil_sweeps is not None else (5 if heavy else 20)
    r_states = []
    for st in range(n_states):  # equilibrate the synthetic walkers of every state (untimed): sweeps x 10 Metropolis sub-steps
        r = torch.as_tensor(r_np[st], dtype=tdt, device=dev)
        eng = ansatz.engine_for(hamil, params_all[st])
        sign, log = eng.wf_forward(r, R)
        state = dict(r=r.clone(), sign=sign, log=log, age=torch.zeros(B, dtype=torch.int32, device=dev),
                     tau=torch.tensor([0.5], dtype=tdt, device=dev))
        for it in range(n_equil):
            eng.mcmc_sweep(state, R, 10, seed=parallel.rank_seed(7 + st), step0=10 * it, walker_offset=rank * B)
        r_states.append(state['r'].clone())
    r = r_states[0]
    eng = ansatz.engine_for(hamil, params)
    pcs = [PhysicalConfiguration(R, rs, torch.zeros(B, device=dev)) for rs in r_states]
    pc = pcs[0]
    loc_ene = hamil.local_energy(ansatz.apply)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)  # > 126 MB L2

    n_sub = wl.get('mcmc_substeps', 0)
    smp_state = None
    if n_sub:  # evaluation step: the walkers are decorrelated by n_sub Metropolis sub-steps before every E_loc (one state)
        sign0, log0 = eng.wf_forward(r, R)
        smp_state = dict(r=r.clone(), sign=sign0, log=log0, age=torch.zeros(B, dtype=torch.int32, device=dev),
                         tau=torch.tensor([0.5], dtype=tdt, device=dev))

    last = {}  # what the most recent step() handed back, by reference: --dump-outputs copies it after the timed loop

    def step(seed, pcs_=None):
        pcs_ = pcs_ or pcs
        if n_sub:
            if pcs_ is not pcs:  # e2e leg: host walkers -> sampler state (psi re-evaluated), as a restart from a checkpoint would
                smp_state['r'].copy_(pcs_[0].r)
                smp_state['sign'], smp_state['log'] = eng.wf_forward(smp_state['r'], R)
            eng.mcmc_sweep(smp_state, R, n_sub, seed=parallel.rank_seed(11), step0=n_sub * (1000 + seed), walker_offset=rank * B)
            pcs_ = [PhysicalConfiguration(R, smp_state['r'], torch.zeros(B, device=dev))]
        Es, sts = [], []
        for st in range(n_states):
            E, stt = loc_ene(seed, params_all[st], pcs_[st])
            Es.append(E); sts.append(stt)
        last.update(r=[p_.r for p_ in pcs_], E=Es, stats=sts)
        if n_states > 1:  # pairwise overlap penalty: every state's wave function on every state's walkers (loss/overlap.py:19-150)
            from deepqmc_b200.overlap import compute_mean_overlap, compute_psi_ratio

            pc_all = PhysicalConfiguration(R, torch.stack([p_.r for p_ in pcs_]), torch.zeros(n_states, B, device=dev))
            ratio, _ = compute_psi_ratio(ansatz, params_all, pc_all)
            last['overlap'] = compute_mean_overlap(ratio)
            E = torch.cat(Es)
            return parallel.energy_statistics(E, {k: torch.cat([s_[k] for s_ in sts]) for k in sts[0]}), E
        return parallel.energy_statistics(Es[0], sts[0]), Es[0]

    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()  # started before the warm-up: NVML start-up must not overlap the timed region
    for w in range(a.warmup):
        step(w)
    torch.cuda.synchronize()
    if world > 1:
        torch.distributed.barrier()
    clocks.rows.clear()  # keep only the samples taken during the timed region
    l0 = eng.launch_count
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.steps)]
    torch.cuda.synchronize()
    t_wall0 = time.perf_counter()
    for s in range(a.steps):
        flush.zero_()  # L2 flush between timed iterations (outside the per-step events)
        evs[s][0].record()
        stats, E = step(100 + s)
        evs[s][1].record()
    torch.cuda.synchronize()
    if world > 1:
        torch.distributed.barrier()
    t_wall = time.perf_counter() - t_wall0
    launches = eng.launch_count - l0
    clk = clocks.stop() if rank == 0 else None
    if a.dump_outputs and rank == 0:  # before the e2e leg: the sampler state of lih_eval_step moves on in place
        per_walker = {'walkers': torch.cat(last['r']), 'E_loc': torch.cat(last['E'])}
        per_walker.update({k.replace('/', '_'): torch.cat([s_[k] for s_ in last['stats']]) for k in last['stats'][0]})
        other = {'stat_' + k.replace('/', '_'): v for k, v in stats.items()}
        if 'overlap' in last:
            other.update(overlap_loss=last['overlap'][0], overlap=last['overlap'][1]['overlap/pairwise/mean'])
        dump_outputs(a.dump_outputs, per_walker, other)
    per_step = [e0.elapsed_time(e1) for e0, e1 in evs]
    ms = torch.tensor([sum(per_step)], device=dev, dtype=torch.float64)
    if world > 1:
        torch.distributed.all_reduce(ms, op=torch.distributed.ReduceOp.MAX)
    total_ms = ms.item()
    value = n_states * B * world * a.steps / (total_ms / 1e3)

    # ---- e2e: host buffers through the plugin API, H2D + D2H inside the timed region ----------
    r_host = [rs.cpu().pin_memory() for rs in r_states]
    R_host = R.cpu().pin_memory()
    def e2e_step(seed):
        Rd = R_host.to(dev, non_blocking=True)
        pcs_h = [PhysicalConfiguration(Rd, rh.to(dev, non_blocking=True), torch.zeros(B, device=dev)) for rh in r_host]
        _, E = step(seed, pcs_h)
        return E.cpu()
    # long steps (seconds): the pipeline is warm already, bound the e2e leg to a few steps
    # (same number of steps as the device-timed leg unless that would take more than ~2 minutes; never more than --steps)
    slow = total_ms / a.steps > 500.0
    e2e_warm, e2e_steps = (1, min(a.steps, max(3, int(120e3 / (total_ms / a.steps))))) if slow else (3, a.steps)
    for w in range(e2e_warm):
        e2e_step(w)
    torch.cuda.synchronize()
    if world > 1:
        torch.distributed.barrier()
    t0 = time.perf_counter()
    for s in range(e2e_steps):
        e2e_step(s)
    torch.cuda.synchronize()
    te = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
    if world > 1:
        torch.distributed.all_reduce(te, op=torch.distributed.ReduceOp.MAX)
    e2e_val = n_states * B * world * e2e_steps / te.item()
    esz = r_host[0].element_size()

    # ---- roofline of the dominant kernel (dense-layer GEMMs), timed live with CUDA events ------
    roof = None
    if rank == 0:
        n_prof = 1 if slow else 3
        eng.profile_begin()
        for s in range(n_prof):
            for st in range(n_states):
                loc_ene(s, params_all[st], pcs[st])  # rank-local: no collective here (the other ranks are already done)
        cls = eng.profile_end_classes()  # {class: (ms, algorithmic flops, launches)} of the tensor-core kernels, timed live
        gemm_ms = sum(v[0] for v in cls.values())
        n_gemm = sum(v[2] for v in cls.values())
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
        except Exception:
            pass
        peak = peaks.get('bf16_tflops_sustained', 1590.0 * 0.88)
        dom = max(cls, key=lambda k: cls[k][0])  # the class the step spends most time in
        dms, dfl, dn = cls[dom]
        achieved = dfl / (dms * 1e-3) / 1e12 if dms > 0 else 0.0
        names = {'row_gemm': 'dense-layer row GEMM (' + ('tc::gemm3xtf32_kernel, tcgen05 3xTF32' if backend else 'CUDA-core gemm_kernel') + ')',
                 'mlp_block': 'fused MLP block (tc::mlp_block_f16_kernel, tcgen05 3xFP16)',
                 'trunk': 'whole-trunk kernel (tc::trunk_f16_kernel: all layers, dense GEMMs + attention, tcgen05 3xFP16, '
                          'one persistent launch per forward chunk)'}
        traffic = TRAFFIC.get(a.workload) if dom == 'trunk' else None
        step_ms = total_ms / a.steps
        roof = {'bound': 'tensor', 'kernel': names[dom], 'achieved': achieved,
                'peak': peak, 'unit': 'TFLOP/s', 'frac': achieved / peak,
                'peak_source': 'MEASURED_PEAKS.json bf16_tflops_sustained' if peaks else 'fallback',
                'scheme_ceiling_frac': 1.0 / 3.0,  # fp32-class accuracy = 3 half-precision products per multiply-add
                'traffic': (traffic or {}).get('bytes_per_launch'), 'traffic_detail': traffic,
                'kernel_share_of_step': (dms / n_prof) / step_ms,
                'kernel_launches_per_step': dn // n_prof,
                'classes': {k: {'ms_per_step': v[0] / n_prof, 'share_of_step': (v[0] / n_prof) / step_ms,
                                'tflops': (v[1] / (v[0] * 1e-3) / 1e12 if v[0] > 0 else None), 'launches_per_step': v[2] // n_prof}
                            for k, v in cls.items()},
                'gemm_share_of_step': (gemm_ms / n_prof) / step_ms,
                'gemm_launches_per_step': n_gemm // n_prof,
                'algorithmic_flops_per_eloc': algorithmic_flops_per_eloc(N, M, n_ecp=n_ecp) if wl['kind'] == 'psiformer' else None,
                'whole_step_tflops': (algorithmic_flops_per_eloc(N, M, n_ecp=n_ecp) * B * a.steps / (total_ms / 1e3) / 1e12
                                      if wl['kind'] == 'psiformer' else None)}
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()
    if rank != 0:
        return 0
    cpu = None
    if not a.no_cpu_baseline and world == 1:
        # the CPU leg runs in a fresh process (fork-based worker pool; this process holds a CUDA context)
        try:
            cp = subprocess.run([sys.executable, os.path.abspath(__file__), '--impl', 'reference', '--workload', a.workload,
                                 '--steps', '2', '--warmup', '1'], capture_output=True, text=True, timeout=1200)
            cpu = json.loads(cp.stdout.strip().splitlines()[-1])['cpu_baseline']
        except Exception as exc:  # the baseline is a reported number, never the thing measured
            cpu = {'value': None, 'unit': unit, 'cores': os.cpu_count(), 'kind': 'port', 'sample': f'failed: {exc!r}'}
    out = {
        'metric': metric, 'value': value, 'unit': unit, 'n_gpus': world, 'steps': a.steps, 'warmup': a.warmup,
        'ms_per_step': total_ms / a.steps, 'ms_per_step_min': min(per_step), 'ms_per_step_median': float(np.median(per_step)),
        'higher_is_better': True, 'scaling': a.scaling, 'vs_baseline': None,
        'dtype': 'f32' if a.dtype == 'float32' else 'f64', 'data': 'synthetic',
        'config': {'workload': workload_name, 'global_batch': B * world, 'walkers_per_gpu': B, 'electronic_states': n_states,
                   'parallelism': f'walker-shard x{world}',
                   'l2': 'flushed between timed iterations (256 MiB memset) and activations >> L2',
                   'step': (f'{n_sub} Metropolis sub-steps (all-electron proposals, in-kernel Philox) + ' if n_sub else '')
                           + 'E_loc of all walkers (+ one all_gather of the packed statistics for N>1)',
                   'gemm_backend': 'tcgen05 (3xFP16 whole-trunk kernel for plain forwards, 3xTF32 row GEMMs for the forward-Laplacian rows)' if backend else 'cuda-core'},
        'clocks': clk, 'e2e': {'value': e2e_val, 'unit': unit, 'h2d_bytes_per_step': (n_states * B * N * 3 + M * 3) * esz,
                               'd2h_bytes_per_step': n_states * B * esz, 'steps': e2e_steps},
        'gpu_launches': int(launches), 'roofline': roof, 'cpu_baseline': cpu,
        'energy_mean': float(stats['energy/mean']), 'wall_s_timed_region': t_wall,
    }
    if n_sub:  # the reference's published proxy is a step RATE (it/s, other hardware: RTX 3090)
        out['it_per_s'] = 1e3 / (total_ms / a.steps)
        out['published_reference'] = {'it_per_s': wl['published_it_per_s'], 'hardware': '1x RTX 3090 (JAX, fp32)',
                                      'source': 'doc/examples/ground_state_lih.ipynb:227,238 (BASELINE.md 1)'}
        out['vs_baseline'] = out['it_per_s'] / wl['published_it_per_s']
    print(json.dumps(out))
    return 0


if __name__ == '__main__':
    sys.exit(main())
