"""Benchmark of the GCC-NMF separation hot path on B200 (contract: see the task statement).

Workload (`config.workload`): BASELINE.json configs[1] -- offline enhancement of synthetic 30 s
stereo @ 16 kHz, 1024-FFT, hop 256, K=1024 atoms, 64 TDOAs, 100 KL-NMF iterations: 1872 stereo
STFT frames per 30 s clip.  A "step" is one pass of the whole pipeline (STFT -> GCC-PHAT angular
spectrogram -> KL-NMF -> all-TDOA GCC-NMF argmax mask -> masked reconstruction -> iSTFT) over one clip.

  value  frames/s with the clip already resident in HBM (CUDA events around each step)
  e2e    frames/s through the public host-buffer call (`GCCNMFPipeline.enhance_host`): pinned host
         samples -> H2D -> pipeline -> D2H of the separated signals, all inside the timed region
  N > 1  one long recording of N x 30 s, frame-sharded over the ranks, ONE dictionary learnt jointly
         (an all-reduce of the (F x K + K) W-update numerator per KL-NMF iteration); weak scaling.

`--impl reference` times the reference's own CPU algorithm (the numpy oracle port: the reference is
pure Python and /root/reference does not exist on the GPU box) on this box's host cores, on the same
30 s clip per step, BLAS threads pinned and recorded, steps bounded by a time budget.

`--dump-outputs DIR` writes what the last timed step returned (on rank 0) as DIR/<name>.npy, so that two builds can be
compared output for output on the same seeded inputs.
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

CFG = dict(sampleRate=16000, windowSize=1024, hopSize=256, dictionarySize=1024, numTDOAs=64,
           numIterations=100, microphoneSeparationInMetres=0.1, duration_s=30.0)
# dram__bytes_read.sum + dram__bytes_write.sum of the five kernels of one KL-NMF iteration (profiles/r02k_ncu_full_nmf_kernels.csv,
# ncu --set full --cache-control none inside the running loop: 39.4 MB of it is the H update re-reading / writing back G^T)
NMF_ITERATION_DRAM_BYTES = 39.7e6
# tensor-core products executed per algorithmic product, averaged over the four contractions of an iteration: (4 + 3 + 4 + 3) / 4
EXECUTED_PRODUCTS = 3.5
METRIC = 'STFT frames/sec (1024-FFT, K=1024) full GCC-NMF pipeline'
UNIT = 'frames/s'
DUMP_LIMIT_BYTES = 64 * 1000 * 1000


def workload_config(n_gpus):
    return {'workload': 'BASELINE.json configs[1]: offline enhancement, synthetic 30 s stereo @16 kHz per GPU, '
                        '1024-FFT hop=256, K=1024, 64 TDOAs, 100 KL-NMF iterations (1872 frames per clip)',
            'frames_per_step': 1872 * n_gpus, 'sharding': 'frames' if n_gpus > 1 else 'none',
            'l2': 'L2 flushed (256 MiB write) between timed steps, flush excluded from the step events',
            'nmf_init': 'seeded numpy draw (gccNMFFunctions.py:70-73) made once per shape at plan time, copied on device per step'}


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler(object):
    FIELDS = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
              'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(index), '--query-gpu=' + self.FIELDS,
                                          '--format=csv,noheader,nounits', '-lms', '20'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')] + [time.perf_counter()])

    def wait_first_row(self, timeout=5.0):
        """nvidia-smi takes a few hundred ms to print its first sample: block until it has."""
        t0 = time.perf_counter()
        while self.proc is not None and not self.rows and time.perf_counter() - t0 < timeout:
            time.sleep(0.01)

    def mark(self):
        return time.perf_counter()

    def stop(self, windows=None):
        """windows: [(t0, t1), ...] perf_counter intervals of the timed regions; only samples inside them are used."""
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        rows = self.rows
        if windows:
            inside = [r for r in rows if any(t0 <= r[-1] <= t1 + 0.05 for t0, t1 in windows)]
            rows = inside or rows
        for r in rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(names, r[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        # under-load samples: the upper half of the observed SM clocks
        sm.sort()
        load = sm[len(sm) // 2:] if sm else []
        return {'sm_mhz': float(np.median(load)) if load else None, 'sm_max_mhz': max(mx) if mx else None,
                'samples': len(sm), 'reasons': sorted(reasons)}


# ------------------------------------------------------------------------------------------------ CPU baseline
def cpu_model():
    try:
        for line in open('/proc/cpuinfo'):
            if line.startswith('model name'):
                return line.split(':', 1)[1].strip()
    except OSError:
        pass
    return 'unknown'


def blas_thread_limit():
    """Threads given to the BLAS pool for the CPU arm: GCCNMF_CPU_THREADS, else every core the pool can use (OpenBLAS builds cap it, 64 here)."""
    env = os.environ.get('GCCNMF_CPU_THREADS')
    return int(env) if env else (os.cpu_count() or 1)


def cpu_baseline(sample_seconds=3.0, repeats=1):
    """The oracle port of the reference numpy path (offlineSpeechEnhancement.ipynb cells 12-41 order)
    timed on this box's host cores on a bounded sample of the same workload, BLAS threads pinned and recorded."""
    from oracle import gccnmf_oracle as orc
    from gcc_nmf_b200.synth import synthetic_stereo
    from threadpoolctl import threadpool_info, threadpool_limits
    x = synthetic_stereo(CFG['duration_s'])[:, :int(sample_seconds * CFG['sampleRate'])]
    frames = 1 + (x.shape[1] - CFG['windowSize']) // CFG['hopSize']
    best, stages = None, None
    with threadpool_limits(limits=blas_thread_limit()):
        blas = sorted({(i.get('internal_api'), i.get('num_threads')) for i in threadpool_info()})
        for _ in range(repeats):
            tm = {}
            t0 = time.perf_counter()
            orc.runEnhancement(x, CFG['sampleRate'], CFG['windowSize'], CFG['hopSize'], CFG['numTDOAs'],
                               CFG['microphoneSeparationInMetres'], CFG['dictionarySize'], CFG['numIterations'], timings=tm)
            dt = time.perf_counter() - t0
            if best is None or dt < best:
                best, stages = dt, tm
    threads = max([n for _, n in blas] or [1])
    return {'value': frames / best, 'unit': UNIT, 'cores': int(min(threads, os.cpu_count() or threads)), 'kind': 'port',
            'sample': '%.1f s of the same synthetic clip (%d frames), same N/hop/K/D/iterations; %.2f s of CPU work; '
                      'numpy %s, BLAS pools %s, %d logical CPUs, %s' % (sample_seconds, frames, best, np.__version__, blas, os.cpu_count() or 0, cpu_model()),
            'seconds': best, 'frames': frames, 'logical_cpus': os.cpu_count(), 'cpu_model': cpu_model(), 'blas_pools': [list(b) for b in blas],
            'stage_seconds': {k: round(v, 3) for k, v in stages.items()}}


REFERENCE_ARM_BUDGET_S = float(os.environ.get('GCCNMF_REFERENCE_BUDGET_S', '300'))


def run_reference(args):
    """`--impl reference`: the reference's own CPU algorithm (the numpy oracle port: the reference is pure Python and does not
    travel to the GPU box) on the SAME workload as the GPU arm -- every step is the whole 30 s clip (1872 frames).  One step
    is ~30 s of host work, so the number of steps actually executed is bounded by a time budget (GCCNMF_REFERENCE_BUDGET_S,
    default 300 s: one warm-up + as many timed steps as fit, at least one); `steps` reports what ran, `steps_requested` what was asked."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    t_start = time.perf_counter()
    vals = []
    warm = cpu_baseline(CFG['duration_s']) if args.warmup > 0 else None      # thread pools, page cache
    est = warm['seconds'] if warm else 40.0
    while len(vals) < max(1, args.steps):
        if vals and time.perf_counter() - t_start + est > REFERENCE_ARM_BUDGET_S:
            break
        vals.append(cpu_baseline(CFG['duration_s']))
        est = vals[-1]['seconds']
    v = [b['value'] for b in vals]
    sec = [b['seconds'] for b in vals]
    b = vals[int(np.argsort(sec)[len(sec) // 2])]                # the median step
    value = float(np.median(v))
    print(json.dumps({
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': len(vals), 'steps_requested': args.steps,
        'warmup': 1 if warm else 0, 'ms_per_step': float(np.median(sec)) * 1e3, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32', 'data': 'synthetic', 'config': workload_config(1),
        'value_min': float(min(v)), 'value_max': float(max(v)), 'value_median': value,
        'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': b['cores'], 'kind': 'port', 'sample': b['sample'],
                         'logical_cpus': b['logical_cpus'], 'cpu_model': b['cpu_model'], 'blas_pools': b['blas_pools'],
                         'stage_seconds': b['stage_seconds']},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}))


# ------------------------------------------------------------------------------------------------ GPU arm
def host_outputs(r):
    """The public entries of a step's result dict copied to the host: complex tensors as (..., 2) real / imaginary pairs in
    their own precision, float64 kept, integers as float64 (exact), everything else float32.  Above DUMP_LIMIT_BYTES in all,
    every array is reduced to the same fixed stride of its flattened elements."""
    import torch
    out = {}
    for name, v in r.items():
        if name.startswith('_'):
            continue
        t = torch.as_tensor(v).detach().cpu()
        if t.is_complex():
            t = torch.view_as_real(t)
        dtype = torch.float64 if t.dtype == torch.float64 or not t.is_floating_point() else torch.float32
        out[name] = t.to(dtype).contiguous().numpy()
    stride = -(-sum(a.nbytes for a in out.values()) // DUMP_LIMIT_BYTES)
    if stride > 1:
        out = {name: np.ascontiguousarray(a.ravel()[::stride]) for name, a in out.items()}
    return out


def write_outputs(directory, outputs):
    os.makedirs(directory, exist_ok=True)
    for name, a in outputs.items():
        np.save(os.path.join(directory, name + '.npy'), a)


def load_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get('bf16_tflops_sustained', d.get('bf16_tflops')), d.get('hbm_gbs'), 'measured (MEASURED_PEAKS.json, sustained bf16)'
    return 1400.0, 6650.0, 'fallback (B200_PROFILING.md)'


def run_gpu(args):
    import torch
    import torch.distributed as dist
    from gcc_nmf_b200.synth import synthetic_stereo

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if args.gpus != world:
        if world == 1 and args.gpus > 1:
            raise SystemExit('launch with torch.distributed.run --nproc-per-node %d for --gpus %d' % (args.gpus, args.gpus))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))

    frames_per_clip = 1 + (int(CFG['duration_s'] * CFG['sampleRate']) - CFG['windowSize']) // CFG['hopSize']
    if world == 1:
        from gcc_nmf_b200.pipeline import GCCNMFPipeline
        pipe = GCCNMFPipeline(CFG['sampleRate'], CFG['windowSize'], CFG['hopSize'], CFG['numTDOAs'],
                              CFG['microphoneSeparationInMetres'], CFG['dictionarySize'], CFG['numIterations'], device=local)
        x_host = torch.from_numpy(synthetic_stereo(CFG['duration_s'])).pin_memory()
        # the public one-call API (gccnmf_separate through GCCNMFPipeline.run_fused): target picking on the device, no host
        # synchronisation inside the flow; the staged enhance() -- same kernels, host-side peak picking -- gives the stage breakdown
        step_dev = lambda xd: pipe.run_fused(xd, 0)                                 # noqa: E731
        step_staged = lambda xd: pipe.enhance(xd, collect_stage_times=True)         # noqa: E731
        step_host = lambda out: pipe.run_fused_host(x_host, 0, out)                 # noqa: E731
        total_frames = frames_per_clip
        api = 'GCCNMFPipeline.run_fused / run_fused_host (one gccnmf_separate call per clip)'
    else:
        from gcc_nmf_b200.distributed import ShardedGCCNMFPipeline
        pipe = ShardedGCCNMFPipeline(CFG['sampleRate'], CFG['windowSize'], CFG['hopSize'], CFG['numTDOAs'],
                                     CFG['microphoneSeparationInMetres'], CFG['dictionarySize'], CFG['numIterations'],
                                     device=local, clip_seconds=CFG['duration_s'])
        x_host = torch.from_numpy(pipe.local_samples()).pin_memory()
        step_dev = lambda xd: pipe.enhance(xd)                                      # noqa: E731
        step_staged = lambda xd: pipe.enhance(xd, collect_stage_times=True)         # noqa: E731
        step_host = lambda out: pipe.enhance_host(x_host, out)                      # noqa: E731
        total_frames = pipe.total_frames
        api = 'ShardedGCCNMFPipeline.enhance / enhance_host'

    h = pipe.h
    x_dev = x_host.to(h.device)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=h.device)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput
    sampler = ClockSampler(local) if rank == 0 else None      # started before the warm-up: its first sample takes a while
    torch.cuda.synchronize()
    t_cold = time.perf_counter()
    r = step_dev(x_dev)                  # cold shape: per-shape buffers (cudaMalloc), TMA tensor maps, lazy module load of every kernel
    torch.cuda.synchronize()
    first_call_ms = (time.perf_counter() - t_cold) * 1e3
    for _ in range(max(args.warmup, 3) - 1):
        r = step_dev(x_dev)
    barrier()
    if sampler:
        sampler.wait_first_row()
    windows = []
    launches0 = h.launches
    step_ms, stage_ms = [], {}
    barrier()
    wall0 = time.perf_counter()
    for _ in range(args.steps):
        flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = step_dev(x_dev)
        e1.record()
        e1.synchronize()
        step_ms.append(e0.elapsed_time(e1))
    barrier()
    wall = time.perf_counter() - wall0
    windows.append((wall0, wall0 + wall))
    launches = h.launches - launches0
    # copied now: the result dict holds views of buffers that the later (untimed) calls overwrite
    outputs = host_outputs(r) if args.dump_outputs and rank == 0 else None
    total_ms = torch.tensor([sum(step_ms)], dtype=torch.float64, device=h.device)
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    total_ms = float(total_ms.item())
    value = total_frames * args.steps / (total_ms * 1e-3)

    # ---- stage breakdown: the staged flow (one library call per stage, CUDA events in between), outside the timed regions
    n_staged = 5
    for _ in range(n_staged):
        flush.fill_(1)
        step_staged(x_dev)
        torch.cuda.synchronize()
        for k, v in pipe.stage_times_ms().items():
            stage_ms[k] = stage_ms.get(k, 0.0) + v / n_staged
    barrier()

    # ---- end to end through the host-buffer API
    out_host = None
    for _ in range(max(args.warmup, 3)):
        out_host = step_host(out_host)
    barrier()
    e2e_ms = []
    e2e_wall0 = time.perf_counter()
    for _ in range(args.steps):
        flush.fill_(1)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        out_host = step_host(out_host)
        e1.record()
        e1.synchronize()
        e2e_ms.append(max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3))
    barrier()
    e2e_total = torch.tensor([sum(e2e_ms)], dtype=torch.float64, device=h.device)
    if world > 1:
        dist.all_reduce(e2e_total, op=dist.ReduceOp.MAX)
    e2e_value = total_frames * args.steps / (float(e2e_total.item()) * 1e-3)
    windows.append((e2e_wall0, time.perf_counter()))
    clocks = sampler.stop(windows) if sampler else None      # samples inside the device-resident AND the end-to-end timed regions

    if rank == 0:
        F, K, I = CFG['windowSize'] // 2 + 1, CFG['dictionarySize'], CFG['numIterations']
        T_local = frames_per_clip
        nmf_ms = stage_ms.get('nmf', float('nan'))
        flops_per_iter = 16.0 * F * K * T_local            # 4 GEMMs x 2 F K (2T) per iteration (SURVEY.md 8d)
        achieved = flops_per_iter * I / (nmf_ms * 1e-3) / 1e12
        peak_tf, peak_hbm, peak_src = load_peaks()
        line = {
            'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': max(args.warmup, 3),
            'ms_per_step': total_ms / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f32', 'data': 'synthetic', 'config': dict(workload_config(world), api=api),
            'stage_ms': {k: round(v, 4) for k, v in stage_ms.items()},
            'stage_ms_source': 'staged flow (one library call per stage, CUDA events between stages), %d extra steps outside the timed regions; same kernels as the timed call' % n_staged,
            'collective': getattr(pipe, 'collective', None),
            'wall_s_timed_region': wall, 'gpu_launches': int(launches), 'clocks': clocks, 'first_call_ms': round(first_call_ms, 2),
            'e2e': {'value': e2e_value, 'unit': UNIT, 'h2d_bytes_per_step': int(x_host.numel() * 4),
                    'd2h_bytes_per_step': int(out_host.numel() * 4), 'ms_per_step': float(e2e_total.item()) / args.steps},
            'roofline': {'kernel': 'KL-NMF iteration: tgemm::plane_gemm_kernel x4 (TMA-fed tcgen05.mma kind::f16 over bf16 hi/lo operand planes, '
                                   'float32 TMEM accumulators) + tma_apply_w_kernel, per rank',
                         'bound': 'tensor', 'achieved': achieved, 'peak': peak_tf, 'unit': 'TFLOP/s',
                         'frac': achieved / peak_tf, 'traffic': NMF_ITERATION_DRAM_BYTES, 'peak_source': peak_src,
                         'algorithmic_flops_per_launch_group': flops_per_iter, 'ms_per_iteration': nmf_ms / I,
                         'executed_tensor_tflops': EXECUTED_PRODUCTS * achieved, 'frac_executed': EXECUTED_PRODUCTS * achieved / peak_tf,
                         'note': 'achieved = algorithmic flops (16 F K T per iteration, SURVEY.md 8d) / CUDA-event time of the NMF stage '
                                 'inside the step; float32-level parity needs the hi/lo bf16 split: the two W.H contractions run 2 MMAs of '
                                 'double width per k-step (all 4 hi/lo products), the H-update and W-numerator contractions 3 MMAs '
                                 '(hi.hi + hi.lo + lo.hi), so executed tensor flops are 3.5x the algorithmic ones: frac_executed is the '
                                 'tensor-pipe view; traffic = DRAM bytes per iteration from the ncu --set full capture in profiles/ '
                                 '(--cache-control none: the L2 state of the running loop)'},
        }
        if world == 1 and not args.no_cpu_baseline:
            line['cpu_baseline'] = cpu_baseline(20.0)      # 10-15 s of CPU work on the host cores (bounded sample of the same clip)
        if outputs is not None:
            write_outputs(args.dump_outputs, outputs)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the outputs of the last timed step as DIR/<name>.npy (float32 / float64, at most 64 MB in all)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs writes the outputs of the b200 arm')
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == '__main__':
    main()
