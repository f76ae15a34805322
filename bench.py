#!/usr/bin/env python
"""bench.py -- mocap frames solved/sec (MoSh++ Stage II) on N B200s.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU algorithm (oracle port)

N = 1   workload = the configuration BASELINE.json's north star quotes its target on: ONE 4000-frame SMPL-H sequence
        (V = 6890, 52 joints, 53 markers, fingers on: 111 free variables in Step 2).  A step = one pass of the hot path
        over that sequence: every frame solved by the reference's schedule (Procrustes + 3 dog-legs on a cold start,
        Step 1 + Step 2 dog-legs on every frame).  ``value`` = frames / device time of the kernel (CUDA events on the
        launching stream, inputs resident, L2 flushed between steps).  ``e2e`` = the same through the reference-facing
        plug-in call ``chmosh.mosh_stageii(mocap_fname, cfg, ...)`` by wall clock: file read, per-subject packing,
        model upload, pinned H2D, kernel, D2H, result dictionary.  BASELINE configs[1] (500 frames) rides along as
        ``secondary``, the 32-sequence configs[4] on one GPU as ``c5_one_gpu`` (the strong-scaling base of N > 1).
N > 1   workload = BASELINE configs[4]: 32 SMPL-H sequences x 4000 frames, sharded over the N GPUs (strong scaling on
        the fixed workload): rank 0 owns all observations, NCCL scatter (grouped send/recv), per-rank solves (device
        pointers in and out of the C-ABI), NCCL gather of the result rows to rank 0.  ``value`` = 128000 frames / max
        over ranks of the device time of the rank's solves; ``e2e`` = pinned host buffers on rank 0 -> host results on
        rank 0 by wall clock, scatter and gather inside.

JSON keys follow the driver contract; DESIGN.md section 7 says how each number is obtained.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = 'mocap frames solved/sec (Stage-II)'
UNIT = 'frames/s'
NS_DESC = 'north-star target: one 4000-frame SMPL-H sequence, 53 markers, Stage II, 1 GPU'
C5_DESC = 'BASELINE configs[4]: 32 SMPL-H sequences x 4000 frames, 53 markers, sharded over the GPUs (NCCL scatter / gather)'
C5_SEQUENCES = 32


def algorithmic_bytes(pk, has_velo=True, fingers=True):
    """SURVEY.md 8(d) / BASELINE.md section 3: fp32 bytes of one frame-iteration in the two-kernel
    (materialised J) formulation.  R = residual rows, n = free variables of Step 2."""
    M, n, p_red = pk.n_markers, len(pk.free_step2), pk.p_red
    R = 3 * M + (pk.prior_d + 1 if pk.prior_k else 0) + p_red + (pk.finger_hi - pk.finger_lo if fingers else 0) + 2 * pk.n_dmpl
    b_k1 = 4 * R * (n + 1) + 4 * (n + 3 * M + p_red + 8) + M
    b_k2 = 4 * R * (n + 1) + 4 * (n * (n + 1) // 2 + n)
    return dict(R=R, n=n, B_K1=b_k1, B_K2=b_k2)


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md): one
    `nvidia-smi -lms 100` child process from the warm-up to the end of the end-to-end leg."""

    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap,utilization.gpu')

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                                          '-i', str(self.index), '-lms', '100'], stdout=subprocess.PIPE, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return
        try:
            self.proc.terminate()
            out, _ = self.proc.communicate(timeout=5)
            for line in out.strip().splitlines():
                r = [x.strip() for x in line.split(',')]
                if len(r) >= 7:
                    self.rows.append(r)
        except Exception:
            pass

    def summary(self):
        if not self.rows:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['unavailable']}
        num = lambda s: s.replace('.', '').isdigit()
        busy = [r for r in self.rows if len(r) > 7 and num(r[7]) and float(r[7]) > 0] or self.rows
        sm = sorted(float(r[0]) for r in busy if num(r[0]))
        reasons = []
        for name, col in (('hw_slowdown', 3), ('hw_thermal_slowdown', 4), ('sw_thermal_slowdown', 5), ('sw_power_cap', 6)):
            if any(len(r) > col and r[col].lower().startswith('active') for r in self.rows):
                reasons.append(name)
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': float(self.rows[0][1]) if num(self.rows[0][1]) else None,
                'reasons': reasons, 'samples': len(self.rows), 'samples_under_load': len(busy)}


def make_case(config: str, seq_idx: int, frames=None, tag=''):
    from moshpp_b200 import synth
    d = tempfile.mkdtemp(prefix=f'mosh_bench_{tag}')
    return synth.make_case(d, config, frames=frames, seq_idx=seq_idx)


def dense(case):
    from moshpp_b200.mocap_interface import MocapSession
    mocap = MocapSession(case['mocap_fname'], case['cfg'].mocap.unit)
    return mocap.frames_for_labels(case['latent_labels'], range(len(mocap)))


def blas_threads():
    try:
        from threadpoolctl import threadpool_info
        return max([p.get('num_threads', 1) for p in threadpool_info()] or [1])
    except Exception:
        return os.cpu_count() or 1


def cpu_reference_frames(case, n_frames: int):
    """The reference's CPU algorithm (float64 oracle in reference-cost mode: full mesh + dense 3V x P Jacobian on every
    evaluation, frame-serial, numpy / BLAS on all host cores) over the first n_frames frames of the workload.
    Returns the wall-clock stamp after every solved frame (seconds from the start of the frame loop)."""
    from oracle import stageii
    stamps = []
    t0 = [None]

    def on_frame(fi):
        stamps.append(time.perf_counter())

    t_start = time.perf_counter()
    stageii.mosh_stageii(case['mocap_fname'], case['cfg'], case['markers_latent'], case['latent_labels'],
                         case['betas'], case['marker_meta'], mode='reference_cost', max_frames=n_frames, on_frame=on_frame)
    return np.array(stamps), t_start


def run_reference(args, rank):
    """--impl reference: chumpy / psbody.smpl are absent (SURVEY.md 8(c)), so the reference's own CPU implementation of
    the path is the oracle port in reference-cost mode.  ONE frame-serial solve of the first (W + K) * n frames of the
    same workload as the CUDA arm; step s = frames [s n, (s+1) n).  The cold-start frame (Procrustes + five
    minimisations) therefore lies in the warm-up steps and the timed steps are steady-state frames."""
    if rank != 0:
        return
    try:        # torchrun pins OMP_NUM_THREADS=1; the reference arm may use every host core
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=os.cpu_count())
    except Exception:
        pass
    n_steps = args.warmup + args.steps
    per = max(1, int(round(args.cpu_frames / n_steps)))
    case = make_case('C5', 0, tag='ref_')
    stamps, t_start = cpu_reference_frames(case, n_steps * per)
    edges = np.concatenate([[t_start], stamps])[::per]           # step boundaries
    step_s = np.diff(edges)[args.warmup:args.warmup + args.steps]
    fps = per * len(step_s) / float(step_s.sum())
    cold = float(stamps[0] - t_start)
    workload = NS_DESC if args.gpus == 1 else C5_DESC
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': fps, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': float(step_s.mean()) * 1e3, 'higher_is_better': True,
        'scaling': 'weak' if args.gpus == 1 else 'strong', 'vs_baseline': None,
        'dtype': 'f64', 'data': 'synthetic (seeded procedural SMPL-H model, markers, motion)',
        'config': {'workload': workload, 'frames': 4000, 'markers': 53, 'free_vars': 111,
                   'frames_per_step': per, 'frames_solved': int(n_steps * per)},
        'cpu_baseline': {'value': fps, 'unit': UNIT, 'cores': blas_threads(), 'kind': 'port',
                         'sample': f'frames {args.warmup * per}..{n_steps * per - 1} of the 4000-frame sequence (one frame-serial '
                                   f'solve, {per} frames per step; the cold-start frame, {cold:.1f} s, lies in the warm-up steps), '
                                   'reference-cost mode: full 6890-vertex mesh and dense 20670x156 Jacobian per evaluation; '
                                   'restated reference, not chumpy',
                         'cold_start_frame_s': cold},
        'e2e': {'value': fps, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)


def load_traffic(key):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the Stage-II kernel from this round's
    `ncu --set full` capture of the same workload (profiles/traffic.json), or None."""
    tfile = os.path.join(ROOT, 'profiles', 'traffic.json')
    try:
        t = json.load(open(tfile))
        e = t.get(key)
        if isinstance(e, dict):
            return e.get('dram_bytes_per_launch'), e.get('source')
    except Exception:
        pass
    return None, None


def roofline(ab, builds, useful_builds, ms, traffic_key):
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    peak = float(peaks.get('hbm_gbs', 6650.0))
    per_unit = ab['B_K1'] + ab['B_K2']
    achieved = per_unit * builds / (ms * 1e-3) / 1e9
    useful = per_unit * useful_builds / (ms * 1e-3) / 1e9
    traffic, src = load_traffic(traffic_key)
    return {'bound': 'hbm', 'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak,
            'traffic': traffic, 'traffic_source': src,
            'achieved_useful': useful, 'frac_useful': useful / peak,
            'bytes_per_frame_iteration': per_unit, 'frame_iterations_per_launch': builds,
            'useful_frame_iterations_per_launch': useful_builds,
            'note': 'achieved = (B_K1+B_K2) x frame-iterations executed / kernel time (SURVEY 8(d) effective-bandwidth '
                    'definition of the J-materialising formulation); *_useful counts only the iterations of the emitted '
                    'frames (what the sequential solve needs), i.e. without the warm-up of the time-parallel chunks. The '
                    'fused kernel keeps J on chip: its DRAM traffic is `traffic`. peak: '
                    + ('measured copy bandwidth (MEASURED_PEAKS.json)' if peaks else 'fallback 6650 GB/s')}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--chunk-len', type=int, default=None)
    ap.add_argument('--chunk-warmup', type=int, default=None)
    ap.add_argument('--warmup-full', type=int, default=None)
    ap.add_argument('--precision', default='f32', choices=['f32', 'f64'])
    ap.add_argument('--cpu-frames', type=int, default=50, help='frames of the reference arm (all steps together)')
    ap.add_argument('--cpu-baseline-frames', type=int, default=10, help='frames of the cpu_baseline sample of the CUDA arm')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-secondary', action='store_true', help='N=1: skip the C2 and C5-on-one-GPU legs')
    ap.add_argument('--sequences', type=int, default=C5_SEQUENCES, help='N>1: number of 4000-frame sequences')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='N=1: write the result arrays of the last timed step of the headline workload as DIR/<name>.npy '
                         '(float64, inputs seeded: identical from run to run)')
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == 'ours' else args.warmup

    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    if args.dump_outputs and (args.impl != 'ours' or world > 1):
        raise SystemExit('--dump-outputs writes the outputs of the one-GPU CUDA path (--impl ours, one process)')

    if args.impl == 'reference':
        run_reference(args, rank)
        return

    import torch
    from moshpp_b200 import chmosh

    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a B200: the Stage-II path has no CPU fallback')
    torch.cuda.set_device(local_rank)
    if args.chunk_warmup is None:
        args.chunk_warmup = chmosh.DEFAULT_WARMUP
    if args.warmup_full is None:
        args.warmup_full = chmosh.DEFAULT_WARMUP_FULL
    if world > 1:
        run_sharded(args, rank, local_rank, world)
    else:
        run_single(args)


# ------------------------------------------------------------------------------------------------------------------
# N = 1
# ------------------------------------------------------------------------------------------------------------------
RESULT_ARRAYS = ('fullpose', 'pose', 'trans', 'dmpls', 'markers_sim', 'errs', 'status', 'counters')
DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Writes every array as <out_dir>/<name>.npy, so that two builds can be compared output for output."""
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f'--dump-outputs: {total} bytes of outputs, more than {DUMP_LIMIT_BYTES}')
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f'{name}.npy'), a)


def time_job(model, pk, opts, obs, vis, args, chunk_len, flush, steps, warmup, keep_outputs=False):
    """Device time of `steps` passes of the product's solve on one resident job: the launch over all chunks, the boundary
    check and the repair launches (chmosh.launch_verified), each launch bracketed by CUDA events on the job's stream.
    ``keep_outputs``: also return, as float64 arrays, the result rows of the last timed pass (what job.download() hands
    a caller)."""
    from moshpp_b200 import chmosh, lib
    prec = {'f32': lib.MOSH2_F32, 'f64': lib.MOSH2_F64}[args.precision]
    tol = chmosh.BOUNDARY_TOL['fast']
    F = obs.shape[0]
    extra = chmosh.first_chunk_extra(args.chunk_warmup, args.warmup_full)
    if chunk_len is None:            # the product's own plan (chmosh.mosh_stageii)
        chunk_len = chmosh.plan_chunk_len([F], chmosh.NUM_SMS_B200, args.chunk_warmup, args.warmup_full, first_extra=extra)
    job = model.job(F, opts, chunk_len=chunk_len, chunk_warmup=args.chunk_warmup, warmup_full=args.warmup_full, precision=prec,
                    first_extra=extra)
    job.upload(obs, vis)
    job.sync()
    for _ in range(warmup):
        flush()
        chmosh.launch_verified(job, tol)
    ms, first_ms, launches = [], [], 0
    t0 = time.perf_counter()
    for _ in range(steps):
        flush()                         # outside the CUDA-event brackets of the step
        bad, rep = chmosh.launch_verified(job, tol)
        ms.append(sum(rep['kernel_ms']))
        first_ms.append(rep['kernel_ms'][0])
        launches += len(rep['kernel_ms'])
    wall = time.perf_counter() - t0
    totals = job.totals()
    outputs = None
    if keep_outputs:          # copies: the end-to-end leg below reuses the job's result buffers
        last = job.download()
        outputs = {k: np.array(getattr(last, k), dtype=np.float64) for k in RESULT_ARRAYS}
    # C-ABI job-level end to end: pinned H2D + launches + D2H of all result arrays
    e2e = []
    for i in range(2 + steps):
        t1 = time.perf_counter()
        res, _ = chmosh.solve_verified(job, obs, vis, tol=tol)
        if i >= 2:
            e2e.append(time.perf_counter() - t1)
    solved = int(((res.status & lib.ST_SOLVED) != 0).sum())
    out = dict(ms=float(np.mean(ms)), first_launch_ms=float(np.mean(first_ms)), e2e_job_ms=float(np.mean(e2e)) * 1e3, totals=totals,
               chunks=job.num_chunks, chunk_len=chunk_len, first_extra=extra, solved=solved, wall=wall, flags=int(np.bitwise_or.reduce(res.status)), launches=launches,
               boundary=rep, outputs=outputs)
    job.close()
    return out


def time_plugin(case, args, steps, warmup, chunk_len=None):
    """Wall clock of the reference-facing call chmosh.mosh_stageii (what MoSh.mosh_stageii invokes), per call.  The very
    first call is timed apart with every cache empty (body-model file cache, subject cache, buffer cache): that is what a
    new subject costs; the timed steps are further sequences of the same subject."""
    from moshpp_b200 import chmosh, lib, pack
    chmosh.clear_subject_cache()
    pack.clear_file_cache()
    lib.load_library().mosh2_release_cached_memory()
    ts, cold = [], None
    out = None
    for i in range(1 + warmup + steps):
        t0 = time.perf_counter()
        out = chmosh.mosh_stageii(case['mocap_fname'], case['cfg'], case['markers_latent'], case['latent_labels'], case['betas'],
                                  case['marker_meta'], chunk_len=chunk_len, chunk_warmup=args.chunk_warmup,
                                  warmup_full=args.warmup_full, precision=args.precision)
        dt = time.perf_counter() - t0
        if i == 0:
            cold = dt * 1e3
        elif i > warmup:
            ts.append(dt)
    return float(np.mean(ts)) * 1e3, out, [round(t * 1e3, 1) for t in ts], cold


def run_single(args):
    import torch
    from moshpp_b200 import chmosh, lib, shard

    dev = 0
    flush_buf = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=f'cuda:{dev}')   # > 126 MB L2

    def flush():
        flush_buf.add_(1)
        torch.cuda.synchronize()

    sampler = ClockSampler(dev)
    sampler.start()
    esz = 4 if args.precision == 'f32' else 8

    # ---- headline: one 4000-frame SMPL-H sequence
    case = make_case('C5', 0, tag='ns_')
    pk, opts, flags = chmosh.prepare_stageii(case['cfg'], case['markers_latent'], case['latent_labels'], case['betas'], case['marker_meta'])
    obs, vis = dense(case)
    F = obs.shape[0]
    model = lib.Model(pk, device=dev)
    ns = time_job(model, pk, opts, obs, vis, args, args.chunk_len, flush, args.steps, args.warmup,
                  keep_outputs=bool(args.dump_outputs))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, ns['outputs'])
    chunk_len = ns['chunk_len']
    e2e_ms, out, e2e_each, e2e_cold = time_plugin(case, args, args.steps, 2, chunk_len=args.chunk_len)
    b = out['stageii_debug_details']['b200']
    h2d = b.get('h2d_bytes', obs.size * esz + vis.size)      # (device input adapter: the raw marker table of the file)
    d2h = F * (pk.p_full + pk.p_red + 3 + pk.n_dmpl + 3 * pk.n_markers + 8) * esz + F * 5 * 4
    ab = algorithmic_bytes(pk)
    line = {
        'metric': METRIC, 'value': F / (ns['ms'] * 1e-3), 'unit': UNIT, 'n_gpus': 1, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': ns['ms'], 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': args.precision,
        'data': 'synthetic (seeded procedural SMPL-H model, markers, motion)',
        'config': {'workload': NS_DESC, 'frames': F, 'markers': pk.n_markers, 'free_vars': ab['n'], 'residual_rows': ab['R'],
                   'chunk_len': chunk_len, 'first_chunk_extra': ns['first_extra'], 'chunk_warmup': args.chunk_warmup, 'warmup_full': args.warmup_full,
                   'chunks': ns['chunks'], 'l2': 'flushed between timed steps (256 MiB write)', 'frames_solved': ns['solved'],
                   'frame_iterations_per_step': ns['totals']['builds'],
                   'useful_frame_iterations': ns['totals']['emitted_builds'],
                   'executed_over_useful': ns['totals']['builds'] / max(1, ns['totals']['emitted_builds']),
                   'residual_evals_per_step': ns['totals']['evaluations'], 'status_flags_or': ns['flags'],
                   'launches_per_step': ns['launches'] / args.steps, 'first_launch_ms': ns['first_launch_ms'],
                   'boundary_check': {k: ns['boundary'][k] for k in ('rounds', 'repaired_chunks', 'chunks_over_tol_first',
                                                                     'boundary_delta_first', 'boundary_delta_max', 'unverified_chunks')},
                   'schedule': 'time-parallel chunks, verified: launch over all chunks + boundary check + resume-mode repair '
                               'launches of the chunks whose warm-up left more than the tolerance (all inside ms_per_step)'},
        'roofline': roofline(ab, ns['totals']['builds'], ns['totals']['emitted_builds'], ns['ms'], 'NS'),
        'e2e': {'value': F / (e2e_ms * 1e-3), 'unit': UNIT, 'h2d_bytes_per_step': int(h2d), 'd2h_bytes_per_step': int(d2h),
                'ms_per_step': e2e_ms,
                'what': 'wall clock of chmosh.mosh_stageii(mocap_fname, cfg, ...) per call: mocap file read, label plan, job '
                        'create, pinned H2D of the raw marker table + device-side input adapter, verified launches (the host copy '
                        'of the clean-up and the observation lists are made behind them), D2H, result dictionary; the per-SUBJECT constants (packed model, '
                        'device copy) come from the subject cache after the first call -- first_call_ms is that first call '
                        'with every cache empty (body-model pickle, packing, model upload, buffer allocation)',
                'first_call_ms': e2e_cold, 'subject_cache_hit': b['subject_cache_hit'],
                'kernel_ms_inside': b['kernel_ms'], 'host_ms_last_call': b['host_ms'], 'ms_each_call': e2e_each,
                'c_abi_job_level': {'value': F / (ns['e2e_job_ms'] * 1e-3), 'ms_per_step': ns['e2e_job_ms'],
                                    'what': 'mosh2_job_upload + verified launches + download with host buffers (resident model and job)'}},
        'gpu_launches': ns['launches'],
        'wall_s_timed_region': ns['wall'],
    }
    model.close()

    if not args.no_secondary:
        ksteps = min(args.steps, 5)
        # ---- BASELINE configs[1]: 500 frames
        c2 = make_case('C2', 0, tag='c2_')
        pk2, opts2, _ = chmosh.prepare_stageii(c2['cfg'], c2['markers_latent'], c2['latent_labels'], c2['betas'], c2['marker_meta'])
        o2, v2 = dense(c2)
        m2 = lib.Model(pk2, device=dev)
        r2 = time_job(m2, pk2, opts2, o2, v2, args, None, flush, ksteps, 3)
        m2.close()
        e2, _, _, _ = time_plugin(c2, args, ksteps, 2)
        line['secondary'] = {
            'workload': 'BASELINE configs[1]: SMPL-H 500-frame sequence, 53 markers', 'value': o2.shape[0] / (r2['ms'] * 1e-3),
            'ms_per_step': r2['ms'], 'e2e_value': o2.shape[0] / (e2 * 1e-3), 'e2e_ms_per_step': e2, 'chunks': r2['chunks'],
            'frame_iterations_per_step': r2['totals']['builds'], 'useful_frame_iterations': r2['totals']['emitted_builds'],
            'steps': ksteps}
        # ---- BASELINE configs[4] on ONE GPU (the base of the strong-scaling run at N > 1)
        line['c5_one_gpu'] = c5_local(args, dev, ksteps, flush)

    sampler.stop()
    line['clocks'] = sampler.summary()
    if not args.no_cpu_baseline:
        try:
            from threadpoolctl import threadpool_limits
            threadpool_limits(limits=os.cpu_count())
        except Exception:
            pass
        n = max(2, args.cpu_baseline_frames)
        stamps, t_start = cpu_reference_frames(case, n)
        steady = (n - 1) / float(stamps[-1] - stamps[0])
        line['cpu_baseline'] = {
            'value': steady, 'unit': UNIT, 'cores': blas_threads(), 'kind': 'port',
            'sample': f'frames 1..{n - 1} of the same 4000-frame workload (steady state; frame 0, the cold start with five '
                      f'minimisations, took {stamps[0] - t_start:.1f} s and is reported apart), frame-serial float64 oracle in '
                      'reference-cost mode (full mesh + dense Jacobian per evaluation); restated reference, not chumpy',
            'value_incl_cold_start': n / float(stamps[-1] - t_start)}
    print(json.dumps(line), flush=True)


def c5_inputs(n_seq, pin=True):
    """Observations of n_seq 4000-frame sequences (same subject, model and marker layout; different motion, noise and
    drop-outs per sequence) as float32 / uint8 host tensors."""
    import torch
    from moshpp_b200 import chmosh, synth
    try:        # torchrun pins OMP_NUM_THREADS=1; synthesising the observations is set-up work, let it use the host cores
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=max(1, (os.cpu_count() or 8) // max(1, int(os.environ.get('LOCAL_WORLD_SIZE', '1')))))
    except Exception:
        pass
    d = tempfile.mkdtemp(prefix='mosh_bench_c5_')
    first = synth.make_case(d, 'C5', seq_idx=0)
    pk, opts, _ = chmosh.prepare_stageii(first['cfg'], first['markers_latent'], first['latent_labels'], first['betas'], first['marker_meta'])
    obs_list, vis_list = [], []
    F = first['obs'].shape[0]
    for i in range(n_seq):
        # one subject (betas, markers_latent) across all sequences: new motion / noise / drop-outs per sequence
        pose, trans, dm = synth.make_motion(pk, F, seed=synth.SEED_MOTION + 4 + 1000 * i)
        mk = synth.forward_markers(pk, pose, trans, None)
        nrng = np.random.default_rng(synth.SEED_NOISE + i)
        o = mk + nrng.normal(0.0, 1e-3, mk.shape)
        drng = np.random.default_rng(synth.SEED_DROPOUT + i)
        v = np.ones((F, pk.n_markers), dtype=bool)
        for m in range(pk.n_markers):
            missing = 0
            while missing < 0.03 * F:
                L = int(drng.integers(5, 51))
                s = int(drng.integers(0, F - 1))
                v[s:s + L, m] = False
                missing += L
        o[~v] = 0.0
        ot, vt = torch.from_numpy(o.astype(np.float32)), torch.from_numpy(v.astype(np.uint8))
        obs_list.append(ot.pin_memory() if pin else ot)
        vis_list.append(vt.pin_memory() if pin else vt)
    return pk, opts, obs_list, vis_list


def c5_local(args, dev, steps, flush):
    """All 32 sequences on one GPU (no scatter): the N = 1 point of the strong-scaling series."""
    import torch
    from moshpp_b200 import shard
    pk, opts, obs_list, vis_list = c5_inputs(args.sequences)
    F = [int(o.shape[0]) for o in obs_list]
    solver = shard.GpuRankSolver({i: pk for i in range(len(F))}, opts, dict(enumerate(F)), dev,
                                 chunk_warmup=args.chunk_warmup, warmup_full=args.warmup_full)
    resident = {i: (obs_list[i].cuda(dev), vis_list[i].cuda(dev)) for i in range(len(F))}
    torch.cuda.synchronize()
    ms, e2e = [], []
    for s in range(2 + steps):
        flush()
        solver(resident)
        if s >= 2:
            ms.append(solver.span_ms())
    for s in range(1 + steps):
        t0 = time.perf_counter()
        mine = {i: (obs_list[i].cuda(dev, non_blocking=True), vis_list[i].cuda(dev, non_blocking=True)) for i in range(len(F))}
        rows = solver(mine)
        host = {i: r.cpu() for i, r in rows.items()}
        if s >= 1:
            e2e.append(time.perf_counter() - t0)
    tot = solver.totals()
    out = {'workload': C5_DESC + ' -- all on one GPU', 'value': sum(F) / (np.mean(ms) * 1e-3), 'ms_per_step': float(np.mean(ms)),
           'e2e_value': sum(F) / float(np.mean(e2e)), 'e2e_ms_per_step': float(np.mean(e2e)) * 1e3,
           'chunk_len': solver.chunk_len, 'chunks': solver.num_chunks(), 'frame_iterations_per_step': tot['builds'],
           'useful_frame_iterations': tot['emitted_builds'], 'steps': steps, 'sequences': len(F)}
    solver.close()
    return out


# ------------------------------------------------------------------------------------------------------------------
# N > 1: BASELINE configs[4], strong scaling
# ------------------------------------------------------------------------------------------------------------------
def run_sharded(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    from moshpp_b200 import shard

    os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
    dev = torch.device('cuda', local_rank)
    dist.init_process_group('nccl', device_id=dev)

    def barrier():
        dist.barrier()
        torch.cuda.synchronize()

    def allmax(x):
        t = torch.tensor([float(x)], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    n_seq = args.sequences
    # every rank builds the (small) subject constants itself; only rank 0 owns observations
    if rank == 0:
        pk, opts, obs_list, vis_list = c5_inputs(n_seq)
    else:
        pk, opts, _, _ = c5_inputs(0)
        obs_list = vis_list = None
    F = [4000] * n_seq
    assignment = shard.assign_sequences(F, world)
    mine_ids = assignment[rank]
    solver = shard.GpuRankSolver({i: pk for i in mine_ids}, opts, {i: F[i] for i in mine_ids}, local_rank,
                                 chunk_warmup=args.chunk_warmup, warmup_full=args.warmup_full)
    width = solver.row_width
    flush_buf = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)

    def flush():
        flush_buf.add_(1)
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    sampler.start()
    shapes = [(f, pk.n_markers) for f in F]
    # ---- device-timed leg: this rank's sequences resident on its GPU
    resident = shard.scatter_observations(obs_list, vis_list, assignment, shapes)
    for _ in range(args.warmup):
        flush()
        solver(resident)
    barrier()
    t_wall0 = time.perf_counter()
    dev_ms = []
    launches = 0
    for _ in range(args.steps):
        flush()
        solver(resident)
        dev_ms.append(solver.span_ms())      # CUDA events on the jobs' streams, summed over the launches of the solve
        launches += sum(len(r['kernel_ms']) for r in solver.reports)
    barrier()
    t_wall = time.perf_counter() - t_wall0
    ms_step = allmax(np.mean(dev_ms))
    tot = solver.totals()
    tt = torch.tensor([tot['builds'], tot['emitted_builds'], tot['evaluations'], launches], dtype=torch.float64, device=dev)
    dist.all_reduce(tt)
    launches_total = tt[3].item()
    # ---- e2e: pinned host buffers on rank 0 -> scatter -> solve -> gather -> host results on rank 0
    e2e = []
    for s in range(2 + args.steps):
        barrier()
        t0 = time.perf_counter()
        out, _ = shard.solve_sharded(F, [pk.n_markers] * n_seq, [width] * n_seq, solver, obs_list, vis_list)
        host = {i: r.cpu() for i, r in out.items()}          # rank 0: D2H of every sequence's rows
        torch.cuda.synchronize()
        dt = allmax(time.perf_counter() - t0)
        if s >= 2:
            e2e.append(dt)
    sampler.stop()
    e2e_ms = float(np.mean(e2e)) * 1e3
    total_frames = sum(F)
    if rank == 0:
        solved = sum(int(((r[:, 3 * pk.n_joints + 3 + pk.n_dmpl + 8].numpy().astype(np.int64) & 1) != 0).sum()) for r in host.values())
        ab = algorithmic_bytes(pk)
        h2d = sum(int(o.numel()) * 4 + int(v.numel()) for o, v in zip(obs_list, vis_list))
        d2h = total_frames * width * 4
        builds, useful = int(tt[0].item()), int(tt[1].item())
        line = {
            'metric': METRIC, 'value': total_frames / (ms_step * 1e-3), 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': ms_step, 'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None,
            'dtype': args.precision, 'data': 'synthetic (seeded procedural SMPL-H model, markers, motion)',
            'config': {'workload': C5_DESC, 'sequences': n_seq, 'frames': total_frames, 'markers': pk.n_markers,
                       'free_vars': ab['n'], 'residual_rows': ab['R'], 'sequences_per_gpu': [len(a) for a in assignment],
                       'chunk_len': solver.chunk_len, 'chunks_per_gpu': solver.num_chunks(), 'chunk_warmup': args.chunk_warmup,
                       'warmup_full': args.warmup_full, 'l2': 'flushed between timed steps (256 MiB write)',
                       'frames_solved': solved, 'frame_iterations_per_step': builds, 'useful_frame_iterations': useful,
                       'executed_over_useful': builds / max(1, useful),
                       'collectives': 'grouped NCCL send/recv: scatter of observations from rank 0, gather of result rows to rank 0 '
                                      '(inside e2e; the device-timed value has the observations resident)',
                       'single_gpu_base': 'bench.py --gpus 1 reports the same 32-sequence workload on one GPU under c5_one_gpu'},
            'roofline': roofline(ab, builds / world, useful / world, ms_step, 'C5'),
            'e2e': {'value': total_frames / (e2e_ms * 1e-3), 'unit': UNIT, 'h2d_bytes_per_step': int(h2d), 'd2h_bytes_per_step': int(d2h),
                    'ms_per_step': e2e_ms,
                    'what': 'shard.solve_sharded: pinned host observations on rank 0 -> H2D -> NCCL scatter -> per-rank solves '
                            '(device pointers through the C-ABI) -> NCCL gather -> D2H on rank 0; wall clock, max over ranks'},
            'gpu_launches': int(launches_total),
            'clocks': sampler.summary(),
            'wall_s_timed_region': t_wall,
        }
        print(json.dumps(line), flush=True)
    solver.close()
    dist.destroy_process_group()


if __name__ == '__main__':
    main()
