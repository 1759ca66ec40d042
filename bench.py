#!/usr/bin/env python
"""Benchmark of the DiffSBDD denoising hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference|reference-gpu]
                    [--workload fullatom|ca|inpaint] [--dump-outputs DIR]

metric : ligand atoms/s through the full DDPM sampling loop of the per-GPU batch.
workload (BASELINE.json configs, SURVEY.md §8(d)):
  fullatom  configs[2] (default; configs[3] under torchrun): crossdock_fullatom_cond dims, 500 steps, batch 64/GPU,
            N_L=25, N_P=175 (rho 0.045 A^-3)                      -> 501 denoiser calls per step
  ca        configs[1]: crossdock_ca_cond dims, 500 steps, batch 32, N_L=25, N_P=40 (rho 0.007 A^-3)
  inpaint   configs[4]: ConditionalDDPM.inpaint, full-atom dims, batch 64, 10 of 25 ligand atoms fixed, center='ligand';
            schedule --inpaint-timesteps x --resamplings (script default 50 x 20, inpaint.py:205-206; also 500 x 1)
step   : ONE complete sampling run (``sample_given_pocket`` / ``inpaint``) of the per-GPU batch.
value  : whole-job atoms/s with the inputs already resident in HBM (CUDA events, max over ranks).
e2e    : same metric through the public API from pinned HOST buffers, host->device copies of the inputs and the
         device->host read of the ligands inside the timed region.
--impl reference     : the reference's CPU implementation of the path (oracle port — /root/reference cannot travel to the
                       GPU box), all host threads it can use, bounded sample per step, extrapolated linearly.
--impl reference-gpu : the same ATen op sequence as the reference on the B200 (device='cuda', eager, reference-order DDPM
                       loop): the fair "beat this" number of SURVEY.md §8(d); bounded sample, extrapolated linearly.
--dump-outputs DIR   : b200 arm: after the timed steps, writes what the sampler returned in the last timed step as
                       DIR/<name>.npy (float32, integer arrays as float64; at most 64 MB, else a fixed seeded sample of
                       rows).  The inputs are seeded, so two builds run with the same arguments can be compared output
                       for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from argparse import Namespace

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = 'ligand_atoms_per_sec_500step_ddpm'
UNIT = 'ligand atoms/s'
DUMP_BYTES = 64 * 10**6      # --dump-outputs writes at most this much

WORKLOADS = {
    # name: (BASELINE.json config index, batch, n_lig, n_pocket, density, norm_values, yml, full-atom?)
    'fullatom': (2, 64, 25, 175, 0.045, (1, 4), 'crossdock_fullatom_cond', True),
    'ca': (1, 32, 25, 40, 0.007, (1, 1), 'crossdock_ca_cond', False),
    'inpaint': (4, 64, 25, 175, 0.045, (1, 4), 'crossdock_fullatom_cond', True),
    # the other network widths the reference ships (no BASELINE.json entry: index None): same batch shapes, tensor-core kernels
    # templated on hidden_nf
    'moad': (None, 64, 25, 175, 0.045, (1, 4), 'moad_fullatom_cond', True),       # hidden_nf 192, edge_embedding_dim 8, cut-offs 4 / 7 A
    'moad_ca': (None, 32, 25, 40, 0.007, (1, 4), 'moad_ca_cond', False),          # hidden_nf 128, 5 layers, joint_nf 32, cut-offs 8 A
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=2)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference', 'reference-gpu'])
    ap.add_argument('--workload', default='fullatom', choices=sorted(WORKLOADS))
    ap.add_argument('--batch', type=int, default=None, help='pockets per GPU (default: the workload\'s)')
    ap.add_argument('--n-lig', type=int, default=None)
    ap.add_argument('--n-pocket', type=int, default=None)
    ap.add_argument('--timesteps', type=int, default=500, help='diffusion steps T of the model / sampling run')
    ap.add_argument('--inpaint-timesteps', type=int, default=50, help='inpaint: sub-sampled steps (inpaint.py:206)')
    ap.add_argument('--resamplings', type=int, default=20, help='inpaint: RePaint resamplings (inpaint.py:205)')
    ap.add_argument('--n-fixed', type=int, default=10, help='inpaint: fixed ligand atoms per sample')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--profile-calls', type=int, default=10)
    ap.add_argument('--cpu-sample-seconds', type=float, default=20.0)
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='b200 arm: write the outputs of the last timed step to DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs needs --impl b200')
    _, b, nl, npk, _, _, _, _ = WORKLOADS[args.workload]
    args.batch = b if args.batch is None else args.batch
    args.n_lig = nl if args.n_lig is None else args.n_lig
    args.n_pocket = npk if args.n_pocket is None else args.n_pocket
    return args


def workload(args):
    from diffsbdd_b200.config import FULLATOM_COND, CA_COND
    _, _, _, _, density, norm_values, yml, fullatom = WORKLOADS[args.workload]
    cfg = FULLATOM_COND if fullatom else CA_COND
    if args.workload == 'moad':        # configs/moad_fullatom_cond.yml:30-46
        cfg = cfg.with_(hidden_nf=192, edge_embedding_dim=8, edge_cutoff_pocket=4.0, edge_cutoff_interaction=7.0)
    if args.workload == 'moad_ca':     # configs/moad_ca_cond.yml:30-46
        cfg = cfg.with_(hidden_nf=128, n_layers=5, joint_nf=32, edge_cutoff_pocket=8.0, edge_cutoff_interaction=8.0)
    return cfg, density, norm_values, yml


def denoiser_calls(args):
    """Denoiser calls of one step (one sampling run)."""
    if args.workload == 'inpaint':
        return args.inpaint_timesteps * args.resamplings + 1
    return args.timesteps + 1


def workload_config(args, world=1):
    """The `config` object of the JSON line: identical keys and values in every arm (b200 / reference / reference-gpu)."""
    idx, _, _, _, density, _, yml, _ = WORKLOADS[args.workload]
    if args.workload == 'fullatom' and world > 1:
        idx = 3
    name = {1: 'conditional C-alpha model', 2: 'conditional full-atom model', 3: 'conditional full-atom model, batch split over GPUs',
            4: 'inpainting (ConditionalDDPM.inpaint, fixed-atom mask + resampling), full-atom model',
            None: 'conditional model of another shipped width'}[idx]
    head = f'BASELINE configs[{idx}]' if idx is not None else 'not a BASELINE.json configuration'
    cfg = {'workload': (f'{head}: {name} ({yml}.yml dims), batch {args.batch}/GPU, N_L={args.n_lig}, '
                        f'N_P={args.n_pocket}'),
           'baseline_config_index': idx, 'global_batch': args.batch * world, 'batch_per_gpu': args.batch,
           'n_lig': args.n_lig, 'n_pocket': args.n_pocket, 'pocket_density_per_A3': density,
           'timesteps': args.timesteps, 'denoiser_calls_per_step': denoiser_calls(args)}
    if args.workload == 'inpaint':
        cfg.update({'inpaint_timesteps': args.inpaint_timesteps, 'resamplings': args.resamplings, 'n_fixed': args.n_fixed,
                    'center': 'ligand'})
    # the same text in every arm (the driver compares the `config` objects of the arms); what differs per arm is in `arm`
    cfg.update({'weights': 'synthetic seed 0 (diffsbdd_b200/synthetic.py), random-init of the named architecture',
                'parallelism': (f'dp{world}: contiguous pocket shards per rank (diffsbdd_b200.distributed), no collective inside the '
                                'loop, final all_gather of the ligands; the reference arm runs on rank 0 only'),
                'l2': ('b200 arm: 256 MiB read+write flush before every timed step and e2e step; reference arms: none '
                       '(CPU arm / eager GPU arm whose working set exceeds L2 per call)')})
    return cfg


def hparams(cfg, args, norm_values):
    egnn = Namespace(device='cuda', joint_nf=cfg.joint_nf, hidden_nf=cfg.hidden_nf, n_layers=cfg.n_layers,
                     attention=cfg.attention, tanh=cfg.tanh, norm_constant=cfg.norm_constant,
                     inv_sublayers=cfg.inv_sublayers, sin_embedding=cfg.sin_embedding,
                     normalization_factor=cfg.normalization_factor, aggregation_method=cfg.aggregation_method,
                     edge_cutoff_ligand=cfg.edge_cutoff_ligand, edge_cutoff_pocket=cfg.edge_cutoff_pocket,
                     edge_cutoff_interaction=cfg.edge_cutoff_interaction,
                     reflection_equivariant=cfg.reflection_equivariant, edge_embedding_dim=cfg.edge_embedding_dim)
    diff = Namespace(diffusion_steps=args.timesteps, diffusion_noise_schedule='polynomial_2',
                     diffusion_noise_precision=5.0e-4, diffusion_loss_type='l2', normalize_factors=list(norm_values))
    hist = np.ones((args.n_lig + 2, args.n_pocket + 2)).tolist()
    return dict(outdir=None, dataset='crossdock', datadir=None, batch_size=args.batch, lr=1e-3, egnn_params=egnn,
                diffusion_params=diff, num_workers=0, augment_noise=0, augment_rotation=False, clip_grad=True,
                eval_epochs=1, eval_params=Namespace(), visualize_sample_epoch=1, visualize_chain_epoch=1,
                auxiliary_loss=False, loss_params=Namespace(), mode='pocket_conditioning', node_histogram=hist,
                pocket_representation='full-atom' if WORKLOADS[args.workload][7] else 'CA')


def inpaint_inputs(cfg, args, n_graphs, seed, device='cpu'):
    """SURVEY.md §8(d) config 5: per sample the first n_fixed of the N_L ligand atoms are known (inpaint.py:117-141),
    known coordinates ~ N(0, 1.5^2 A) around the pocket COM (the synthetic pockets are centred), random one-hot types."""
    g = torch.Generator().manual_seed(1000 + seed)
    n = n_graphs * args.n_lig
    x = torch.randn((n, 3), generator=g) * 1.5
    types = torch.randint(0, cfg.atom_nf, (n,), generator=g)
    fixed = torch.zeros(n)
    fixed.view(n_graphs, args.n_lig)[:, :args.n_fixed] = 1
    lig = {'x': x, 'one_hot': torch.nn.functional.one_hot(types, cfg.atom_nf).float(),
           'size': torch.full((n_graphs,), args.n_lig, dtype=torch.int64),
           'mask': torch.repeat_interleave(torch.arange(n_graphs), args.n_lig)}
    return {k: v.to(device) for k, v in lig.items()}, fixed.to(device)


# ---- clocks sampler (B200_PROFILING.md "clocks DURING the timed region") -------------------------------------
class ClockSampler:
    FIELDS = ('uuid,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
              'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
              'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, device):
        self.uuid = None
        try:
            self.uuid = str(torch.cuda.get_device_properties(device).uuid)
        except Exception:
            pass
        self.rows, self.proc, self.thread = [], None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.FIELDS}', '--format=csv,noheader,nounits',
                                          '-lms', '200'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return

        def pump():
            for line in self.proc.stdout:
                self.rows.append(line.strip())
        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, power, reasons = [], None, [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(',')]
            if len(f) < 9:
                continue
            if self.uuid and self.uuid.replace('GPU-', '') not in f[0]:
                continue
            try:
                sm.append(float(f[1])); smax = float(f[2]); power.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[5:9]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        load = [c for c, p in zip(sm, power) if p > 0.5 * max(power)] if power else sm
        return {'sm_mhz': statistics.median(load) if load else None, 'sm_max_mhz': smax,
                'power_w_max': max(power) if power else None, 'samples': len(sm), 'reasons': sorted(reasons)}


def l2_flush(buf):
    buf.add_(1.0)    # read+write 256 MiB > 126 MB L2


def dump_outputs(arrays, out_dir, limit=DUMP_BYTES):
    """Writes every tensor of ``arrays`` to ``out_dir/<name>.npy``: float32 (float64 stays float64, integers become
    float64, exactly).  If together they exceed ``limit`` bytes, each array keeps the same fraction of its rows, picked
    with a fixed seed: the same rows for the same shapes, so that dumps of two runs stay comparable row for row."""
    out = {}
    for name, t in arrays.items():
        a = t.detach().cpu().numpy()
        out[name] = a.astype(np.float64 if a.dtype == np.float64 or a.dtype.kind in 'iub' else np.float32)
    total = sum(a.nbytes for a in out.values())
    budget = limit - 1024 * len(out)           # room for the .npy headers
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        if total > budget and len(a):
            keep = len(a) * budget // total
            a = a[np.sort(np.random.default_rng(0).choice(len(a), keep, replace=False))]
        np.save(os.path.join(out_dir, name + '.npy'), a)


# ---- reference arms: the oracle port of the reference's PyTorch path, on the host cores or eager on the GPU -----------
def _reference_ddpm(args, device):
    from diffsbdd_b200 import synthetic as syn
    from diffsbdd_b200.conditional_model import ConditionalDDPM
    from oracle.cpu_denoiser import OracleDynamics
    cfg, density, norm_values, yml = workload(args)
    sd = syn.synthetic_state_dict(cfg, 0)
    dyn = OracleDynamics(cfg, sd, device=device)
    hist = np.ones((args.n_lig + 2, args.n_pocket + 2)).tolist()
    ddpm = ConditionalDDPM(dynamics=dyn, atom_nf=cfg.atom_nf, residue_nf=cfg.residue_nf, n_dims=3,
                           timesteps=args.timesteps, noise_schedule='polynomial_2', noise_precision=5e-4,
                           loss_type='l2', norm_values=norm_values, size_histogram=hist)
    ddpm.loop_engine = 'eager'          # the reference's own loop: same torch ops, same order, per-step host syncs
    return ddpm.to(device).eval(), dyn, cfg, density


def _reference_run(args, ddpm, cfg, density, nb, sub_steps, device, seed=3):
    """One bounded sample: ``sub_steps`` reverse steps (+ the final p(x|z0) call) of the workload's sampler on the first
    ``nb`` pockets.  Returns seconds."""
    from diffsbdd_b200 import synthetic as syn
    pocket = syn.synthetic_pocket(cfg, [args.n_pocket] * nb, seed=seed, density=density)
    pocket = {k: v.to(device) for k, v in pocket.items()}
    t0 = time.perf_counter()
    if args.workload == 'inpaint':
        lig, fixed = inpaint_inputs(cfg, args, nb, seed, device)
        ddpm.inpaint(lig, pocket, fixed, resamplings=1, timesteps=sub_steps, center='ligand')
    else:
        ddpm.sample_given_pocket(pocket, torch.full((nb,), args.n_lig, dtype=torch.int64, device=device), timesteps=sub_steps)
    if torch.device(device).type == 'cuda':
        torch.cuda.synchronize()
    return time.perf_counter() - t0


class _CpuReference:
    """The CPU port on a BOUNDED sample of the workload: the first ``nb`` pockets of the batch (CPU cost is linear in the
    number of pockets: graphs are independent), 1 reverse step + the final p(x|z0) call per repetition; atoms/s
    extrapolated to the full loop (every denoiser call of the loop has the same cost; the O(N) update/blend ops between
    calls are <1 % of a call on the CPU).  Built once per process; the torch thread count is calibrated once, under a
    time cap (most likely candidates first)."""

    def __init__(self, args, sub_batch=None, calibrate_s=15.0):
        self.args = args
        self.ddpm, self.dyn, self.cfg, self.density = _reference_ddpm(args, 'cpu')
        self.cores = os.cpu_count() or 1
        self.nb = min(sub_batch or 8, args.batch)
        torch.manual_seed(0)
        self.cands = [c for c in (16, 32, 8, 64, self.cores) if c <= self.cores] or [self.cores]
        self.tried = []
        best_t = None
        t_cal0 = time.perf_counter()
        for th in dict.fromkeys(self.cands):
            torch.set_num_threads(th)
            if not self.tried:
                self.one()                                       # first touch: allocator, oneDNN primitives
            t = self.one()
            self.tried.append(th)
            if best_t is None or t < best_t:
                self.threads, best_t = th, t
            if time.perf_counter() - t_cal0 > calibrate_s:
                break
        torch.set_num_threads(self.threads)

    def one(self):                                               # 2 denoiser calls
        return _reference_run(self.args, self.ddpm, self.cfg, self.density, self.nb, 1, 'cpu')

    def sample(self, budget_s):
        args = self.args
        self.dyn.calls = 0
        t0 = time.perf_counter()
        reps = 0
        while reps < 1 or (time.perf_counter() - t0 < budget_s and reps < 50):
            self.one()
            reps += 1
        dt = time.perf_counter() - t0
        per_call = dt / self.dyn.calls
        n_calls = denoiser_calls(args)
        atoms = self.nb * args.n_lig
        return {'value': atoms / (per_call * n_calls), 'unit': UNIT, 'cores': self.threads, 'kind': 'port',
                'sample': (f'oracle port of the reference PyTorch path (oracle/egnn_oracle.py + eager reference-order DDPM '
                           f'loop) on the first {self.nb} of the {args.batch} pockets, {self.dyn.calls} denoiser calls in '
                           f'{dt:.1f} s = {per_call:.2f} s/call, extrapolated x{n_calls} calls; torch threads calibrated '
                           f'over {self.tried} of {self.cores} host cores -> {self.threads}'),
                'seconds_per_denoiser_call': per_call, 'host_cores': self.cores, 'torch_threads': self.threads,
                'sample_pockets': self.nb}, dt, self.dyn.calls


def cpu_reference_sample(args, budget_s, sub_batch=None):
    return _CpuReference(args, sub_batch).sample(0.5 * budget_s)


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    t_all = time.perf_counter()
    ref = _CpuReference(args)
    n_it = args.warmup + args.steps
    # the whole run stays within ~3 minutes: equal shares of what the calibration left, at least one repetition per step
    times, base = [], None
    for i in range(n_it):
        left = 170.0 - (time.perf_counter() - t_all)
        per_step = max(0.0, min(0.5 * args.cpu_sample_seconds, left / max(1, n_it - i)))
        base, dt, calls = ref.sample(per_step)
        if i >= args.warmup:
            times.append(dt)
    cfgj = workload_config(args, int(os.environ.get('WORLD_SIZE', '1')))
    arm = {'what': 'oracle port of the reference PyTorch op sequence on the host cores',
           'reference_sample': 'bounded sample per step, extrapolated: ' + base['sample']}
    line = {'impl': 'reference', 'arm': arm, 'metric': METRIC, 'value': base['value'], 'unit': UNIT, 'n_gpus': args.gpus,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * statistics.mean(times),
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': cfgj, 'cpu_baseline': base,
            'e2e': {'value': base['value'], 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(line), flush=True)


def run_reference_gpu(args):
    """The reference's op sequence (oracle port, device='cuda') inside the reference-order eager loop on ONE B200, full
    batch: ``sub`` reverse steps + the final call per timed step, extrapolated to the full loop."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    if not torch.cuda.is_available():
        print(json.dumps({'impl': 'reference-gpu', 'unavailable': 'no CUDA device'}))
        return
    device = 'cuda:0'
    ddpm, dyn, cfg, density = _reference_ddpm(args, device)
    sub = 20
    torch.manual_seed(0)
    for _ in range(max(1, min(args.warmup, 2))):
        _reference_run(args, ddpm, cfg, density, args.batch, 2, device)
    dyn.calls = 0
    sampler = ClockSampler(torch.device(device))
    sampler.start()
    times = [_reference_run(args, ddpm, cfg, density, args.batch, sub, device) for _ in range(args.steps)]
    clocks = sampler.stop()
    per_call = sum(times) / dyn.calls
    n_calls = denoiser_calls(args)
    value = args.batch * args.n_lig / (per_call * n_calls)
    cfgj = workload_config(args)
    arm = {'what': 'the reference PyTorch op sequence (oracle port) eager on cuda:0',
           'reference_sample': (f'full batch of {args.batch} pockets, {dyn.calls} denoiser calls in {sum(times):.2f} s = '
                                f'{1e3 * per_call:.1f} ms/call (eager ATen ops incl. per-step host syncs), extrapolated x{n_calls} calls')}
    line = {'impl': 'reference-gpu', 'arm': arm, 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': 1, 'steps': len(times),
            'warmup': args.warmup, 'ms_per_step': 1e3 * per_call * n_calls, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic', 'config': cfgj, 'clocks': clocks,
            'ms_per_denoiser_call': 1e3 * per_call,
            'note': 'oracle/egnn_oracle.py restates the reference op for op (bit-identical on CPU); this is that op sequence on cuda:0'}
    print(json.dumps(line), flush=True)


# ---- B200 arm ---------------------------------------------------------------------------------------------------
def run_b200(args):
    import torch.distributed as dist
    from diffsbdd_b200 import synthetic as syn
    from diffsbdd_b200.distributed import sample_given_pocket_sharded, shard_bounds, shard_pocket
    from diffsbdd_b200.lightning_modules import LigandPocketDDPM

    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if world != args.gpus and world > 1:
        raise SystemExit(f'--gpus {args.gpus} but WORLD_SIZE={world}')
    if not torch.cuda.is_available():
        raise SystemExit('bench.py --impl b200 needs a CUDA device (no CPU fallback exists)')
    torch.cuda.set_device(local_rank)
    device = torch.device('cuda', local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=device)

    cfg, density, norm_values, yml = workload(args)
    model = LigandPocketDDPM(**hparams(cfg, args, norm_values))
    model.ddpm.dynamics.load_state_dict(syn.synthetic_state_dict(cfg, 0))
    model.to(device).eval()
    ddpm, dyn = model.ddpm, model.ddpm.dynamics
    B, NL, NP, T = args.batch, args.n_lig, args.n_pocket, args.timesteps
    inpaint = args.workload == 'inpaint'

    # the WHOLE job (B pockets per rank, weak scaling) is described on every rank; each rank samples its contiguous shard
    # (diffsbdd_b200.distributed, SURVEY.md §8(e)).  Shard r of the job is the batch seeded 3 + r.
    parts = [syn.synthetic_pocket(cfg, [NP] * B, seed=3 + r, density=density) for r in range(world)]
    job = {'x': torch.cat([p['x'] for p in parts]), 'one_hot': torch.cat([p['one_hot'] for p in parts]),
           'size': torch.cat([p['size'] for p in parts]),
           'mask': torch.cat([p['mask'] + r * B for r, p in enumerate(parts)])}
    job_dev = {k: v.to(device) for k, v in job.items()}
    n_lig_job = torch.full((B * world,), NL, dtype=torch.int64, device=device)
    lo, hi = shard_bounds(B * world, world, rank)
    pocket_host = {k: v.contiguous().pin_memory() for k, v in shard_pocket(job, lo, hi).items()}
    pocket_dev = {k: v.to(device) for k, v in pocket_host.items()}
    n_lig_host = torch.full((B,), NL, dtype=torch.int64).pin_memory()
    lig_host = fixed_host = lig_dev = fixed_dev = None
    if inpaint:
        lig_host, fixed_host = inpaint_inputs(cfg, args, B, 3 + rank)
        lig_host = {k: v.pin_memory() for k, v in lig_host.items()}
        fixed_host = fixed_host.pin_memory()
        lig_dev = {k: v.to(device) for k, v in lig_host.items()}
        fixed_dev = fixed_host.to(device)
    flush_buf = torch.zeros(64 * 1024 * 1024, dtype=torch.float32, device=device)
    torch.manual_seed(1234 + rank)
    step_no = [0]

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local_rank])
        torch.cuda.synchronize(device)

    def step_device():
        """One sampling run; returns what the caller receives, by name."""
        step_no[0] += 1
        if inpaint:
            out = ddpm.inpaint({k: v.clone() for k, v in lig_dev.items()}, dict(pocket_dev), fixed_dev,
                               resamplings=args.resamplings, timesteps=args.inpaint_timesteps, center='ligand')
            return dict(zip(('xh_lig', 'xh_pocket', 'lig_mask', 'pocket_mask'), out))
        # library path: this rank's shard + the final all_gather of the ligands (the only collective of the path)
        xh_all, sizes_all, local = sample_given_pocket_sharded(ddpm, dict(job_dev), n_lig_job, base_seed=1000 * step_no[0],
                                                               timesteps=T)
        return dict(zip(('xh_lig_all', 'lig_sizes_all', 'xh_lig', 'xh_pocket', 'lig_mask', 'pocket_mask'),
                        (xh_all, sizes_all) + tuple(local)))

    def step_e2e():
        pocket = {k: v.to(device, non_blocking=True) for k, v in pocket_host.items()}
        if inpaint:
            lig = {k: v.to(device, non_blocking=True) for k, v in lig_host.items()}
            fixed = fixed_host.to(device, non_blocking=True)
            xh_lig, _, lig_mask, _ = ddpm.inpaint(lig, pocket, fixed, resamplings=args.resamplings,
                                                  timesteps=args.inpaint_timesteps, center='ligand')
        else:
            n_lig = n_lig_host.to(device, non_blocking=True)
            xh_lig, _, lig_mask, _ = model.generate_ligand_tensors(pocket, n_lig, timesteps=T)
        return xh_lig.cpu(), lig_mask.cpu()

    def timed(fn, k):
        """k steps between two events; returns (max over ranks of the total ms, per-rank total ms list, what the last
        step returned)."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            l2_flush(flush_buf)
            last = fn()
        e1.record()
        torch.cuda.synchronize(device)
        ms = torch.tensor([e0.elapsed_time(e1)], device=device)
        per_rank = [float(ms.item())]
        if world > 1:
            allms = [torch.empty_like(ms) for _ in range(world)]
            dist.all_gather(allms, ms)
            per_rank = [float(m.item()) for m in allms]
        barrier()
        return max(per_rank), per_rank, last

    for _ in range(args.warmup):
        step_device()
    sampler = ClockSampler(device)
    sampler.start()
    ms_total, per_rank_ms, last = timed(step_device, args.steps)
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(last, args.dump_outputs)      # before anything else reuses the sampler's buffers
    clocks_by_rank = None
    if world > 1:      # every rank sampled its own GPU: the per-rank clocks / power / throttle reasons name the limiter of a slow rank
        allc = [None] * world
        dist.all_gather_object(allc, {'rank': rank, 'sm_mhz': clocks.get('sm_mhz'), 'power_w_max': clocks.get('power_w_max'),
                                      'reasons': clocks.get('reasons')})
        clocks_by_rank = allc
    e_last = dyn.last_num_edges
    atoms_per_step = B * NL * world
    value = atoms_per_step * args.steps / (ms_total / 1e3)

    # e2e through the public API with host buffers
    e2e = None
    if not args.no_e2e:
        step_e2e()
        ms_e2e, _, _ = timed(step_e2e, args.steps)
        h2d = sum(v.numel() * v.element_size() for v in pocket_host.values())
        if inpaint:
            h2d += sum(v.numel() * v.element_size() for v in lig_host.values()) + fixed_host.numel() * 4
            api = 'ConditionalDDPM.inpaint(ligand, pocket, lig_fixed [pinned host]->device, ...) -> .cpu()  (inpaint.py:147)'
        else:
            h2d += n_lig_host.numel() * 8
            api = 'LigandPocketDDPM.generate_ligand_tensors(pocket[pinned host]->device, ...) -> .cpu()'
        d2h = B * NL * (3 + cfg.atom_nf) * 4 + B * NL * 8
        e2e = {'value': atoms_per_step * args.steps / (ms_e2e / 1e3), 'unit': UNIT, 'h2d_bytes_per_step': h2d,
               'd2h_bytes_per_step': d2h, 'ms_per_step': ms_e2e / args.steps, 'api': api}

    launches_fwd = dyn.launches_per_forward
    n_calls = denoiser_calls(args)
    per_iter_extra = 2 if inpaint else 1      # fused DDPM update (+ fused RePaint iteration) per reverse step
    gpu_launches = args.steps * (n_calls * launches_fwd + (n_calls - 1) * per_iter_extra)

    # ---- live kernel timing for the roofline: eager forwards with CUDA events on the launch stream ------------
    roof = roof32 = kernel_ms = None
    if rank == 0:
        st = next(iter(ddpm._graph_cache.values())) if ddpm._graph_cache else None
        z = st['z'].clone() if st else None
        pk = st['pocket'].clone() if st else None
        if z is not None:
            t_in = torch.full((B, 1), 0.5, device=device)
            lm, pm = st['lig_mask'], st['pocket_mask']
            with torch.no_grad():
                dyn(z, pk, t_in, lm, pm)
                dyn.set_profiling(True)
                dyn.collect_profile(reset=True)
                for _ in range(args.profile_calls):
                    l2_flush(flush_buf)
                    dyn(z, pk, t_in, lm, pm)
                prof = dyn.collect_profile(reset=True)
                dyn.set_profiling(False)
            E = dyn.last_num_edges
            N, H, L, S = B * (NL + NP), cfg.hidden_nf, cfg.n_layers, cfg.inv_sublayers
            n_gcl = args.profile_calls * L * S
            gcl_ms = prof['edge_gcl']['ms'] / max(1, n_gcl)
            mode = dyn.math_mode
            tensor_path = bool(mode & 2)
            split = '3xfp16' if (mode & 8) else '3xtf32'
            kname = (f'tc_edge_kernel<gcl,{split}>' if tensor_path else f'edge_gcl_kernel<{H}>')
            # algorithmic work of ONE launch of the dominant kernel (DESIGN.md §4): all E edges through the factorised first layer
            # (+SiLU), the HxH second layer, SiLU, attention gate and the receiver segment sum
            alg_bytes = N * 2 * H * 4 + N * H * 4 + E * 12 + N * 16 + (H * H + 7 * H) * 4
            alg_flops = E * (2 * H * H + 12 * H)
            peaks = {}
            try:
                with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
                    peaks = json.load(f)
            except Exception:
                pass
            hbm_peak = float(peaks.get('hbm_gbs', 6650.0))
            tens_peak = float(peaks.get('bf16_tflops', 1590.0))
            src = 'MEASURED_PEAKS.json (of measured)' if peaks else 'B200_PROFILING.md fallback (of fallback)'
            traffic, traffic_src, traffic_edges = None, None, None
            try:   # DRAM bytes per launch from the committed ncu --set full capture (never measured under the profiler here)
                with open(os.path.join(ROOT, 'profiles', 'roofline_traffic.json')) as f:
                    tj = json.load(f)
                # the capture is of the full-atom dimensions (N = 64 x 200 nodes); inpaint runs the same shapes, other workloads have none
                tr = tj.get(f'{kname}@{args.workload}') or (tj.get(kname) if args.workload in ('fullatom', 'inpaint') else None)
                if tr:
                    traffic, traffic_src, traffic_edges = tr['dram_bytes_per_launch'], tr['source'], tr.get('edges')
            except Exception:
                pass
            ach_b = alg_bytes / (gcl_ms * 1e-3) / 1e9
            ach_f = alg_flops / (gcl_ms * 1e-3) / 1e12
            smax = (clocks.get('sm_max_mhz') or 1965.0)
            fp32_peak = torch.cuda.get_device_properties(device).multi_processor_count * 128 * 2 * smax * 1e6 / 1e12
            # the capture's geometry has more edges than this launch: only the 12 B/edge of CSR indices and input distances scale with E
            if traffic is not None and traffic_edges:
                traffic = int(traffic - 12 * (traffic_edges - E))
                traffic_src += f'; captured at E={traffic_edges}, reported for E={E} (-12 B per edge)'
            common = {'kernel': kname, 'avg_launch_ms': gcl_ms, 'edges': E, 'traffic': traffic, 'traffic_edges': traffic_edges,
                      'traffic_source': traffic_src, 'algorithmic_bytes_per_launch': alg_bytes,
                      'algorithmic_flops_per_launch': alg_flops}
            if tensor_path:
                # the contraction runs on the tensor pipe as 3 split products: executed tensor FLOPs = 3 x algorithmic
                roof = dict(common, bound='tensor', achieved=ach_f, peak=tens_peak, unit='TFLOP/s', frac=ach_f / tens_peak,
                            executed_tensor_tflops=3 * ach_f, executed_frac=3 * ach_f / tens_peak,
                            peak_source='bf16_tflops, ' + src,
                            note=('achieved counts ALGORITHMIC fp32 FLOPs (one product per MAC); the kernel executes 3 half-precision '
                                  'MMAs per MAC to keep fp32-grade accuracy, so the tensor pipe does 3x this'))
                roof32 = {'bound': 'hbm', 'kernel': kname, 'achieved': ach_b, 'peak': hbm_peak, 'unit': 'GB/s', 'frac': ach_b / hbm_peak,
                          'peak_source': 'hbm_gbs, ' + src, 'note': 'HBM fraction as BASELINE.json north_star requests; the path is not HBM-bound'}
            else:
                roof = dict(common, bound='hbm', achieved=ach_b, peak=hbm_peak, unit='GB/s', frac=ach_b / hbm_peak,
                            peak_source='hbm_gbs, ' + src,
                            note='kernel is FP32-FMA bound by construction at hidden_nf=256 (SURVEY.md §8(d)); see roofline_fp32')
                roof32 = {'bound': 'fp32_simt', 'kernel': kname, 'achieved': ach_f, 'peak': fp32_peak, 'unit': 'TFLOP/s',
                          'frac': ach_f / fp32_peak, 'peak_source': f'SMs x 128 FMA x 2 x clocks.max.sm ({smax:.0f} MHz), nominal'}
            tot = sum(v['ms'] for v in prof.values())
            kernel_ms = {k: round(v['ms'] / args.profile_calls, 4) for k, v in prof.items()}
            kernel_ms['total_per_call'] = round(tot / args.profile_calls, 4)

    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_base, _, _ = cpu_reference_sample(args, args.cpu_sample_seconds)

    if rank == 0:
        cfgj = workload_config(args, world)
        engine = 'eager'
        if ddpm._graph_cache:
            engine = ('cuda_graph replay: denoiser + fused reverse update + fused RePaint iteration per (s, u)' if inpaint
                      else 'cuda_graph replay of one reverse step')
        arm = {'what': 'diffsbdd_b200 (sm_100a kernels through the C ABI)',
               'arithmetic': {0: 'fp32 FFMA', 7: '3xTF32 tcgen05', 15: '3xFP16 tcgen05'}.get(dyn.math_mode, str(dyn.math_mode)),
               'edges_last_call': e_last, 'loop_engine': engine}
        per_rank_step = [m / args.steps for m in per_rank_ms]
        line = {'arm': arm, 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
                'warmup': args.warmup, 'ms_per_step': ms_total / args.steps, 'higher_is_better': True,
                'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic', 'config': cfgj,
                'ms_per_step_by_rank': {'min': min(per_rank_step), 'median': statistics.median(per_rank_step),
                                        'max': max(per_rank_step)},
                'clocks': clocks, 'clocks_by_rank': clocks_by_rank, 'e2e': e2e, 'gpu_launches': gpu_launches,
                'launches_per_denoiser_call': launches_fwd, 'math_mode': dyn.math_mode, 'roofline': roof, 'roofline_secondary': roof32,
                'kernel_ms_per_denoiser_call': kernel_ms, 'cpu_baseline': cpu_base}
        if inpaint:
            gen = (NL - args.n_fixed) / NL
            line['generated_atoms_per_s'] = value * gen        # atoms actually generated (N_L - n_fixed per sample)
            if e2e:
                e2e['generated_atoms_per_s'] = e2e['value'] * gen
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == 'reference':
        run_reference(args)
    elif args.impl == 'reference-gpu':
        run_reference_gpu(args)
    else:
        run_b200(args)


if __name__ == '__main__':
    main()
