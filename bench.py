#!/usr/bin/env python
"""Benchmark of the DynaBOA per-frame hot path: adapted frames/sec on the synthetic 3DPW-shape stream.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2|c3|c5] [--dump-outputs DIR]

One "step" = one adapted frame at BASELINE.json configs[1] (C2: 1 inner step, batch 1; S-adapt scope of
SURVEY.md §8d: adaptation + one output forward/SMPL).  Prints ONE JSON line (see DESIGN.md "Measurement").
``--impl reference`` times the CPU oracle port of the reference path on the host cores (the reference itself
cannot travel to the GPU box and has no importable package; see oracle/__init__.py).
"""
import argparse
import gc
import json
import os
import subprocess
import sys
import shutil
import tempfile
import threading
import time
from types import SimpleNamespace

import numpy as np
import torch

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

METRIC = 'adapted frames/sec (224x224, 1 inner step)'
WORKLOADS = {
    'c2': dict(inner_step=1, retrieval=0, lower_level_mixtrain=0, upper_level_mixtrain=0, dynamic_boa=0, sample_num=1),
    'c3': dict(inner_step=3, retrieval=1, lower_level_mixtrain=1, upper_level_mixtrain=1, dynamic_boa=0, sample_num=8),
    # BASELINE.json configs[4]: C3 + the dynamic re-adaptation loop at the reference's threshold (dynaboa_benchmark.py:48-49); the
    # trip count is data dependent; under torchrun the (a.b, |a|^2, |b|^2) sums are all-reduced so that every rank takes the same one
    # The reference threshold 3.1e-4 never fires on the seeded random weights of the synthetic stream (1 - cos of feature 12 after one
    # outer step is 5e-6 .. 9e-5 there, profiles/r02_summary.md); 2e-5 sits inside that distribution, so the trip counts are mixed
    # (0..8 per frame), which is what configs[4] asks to exercise.  --cos-threshold overrides.
    'c5': dict(inner_step=3, retrieval=1, lower_level_mixtrain=1, upper_level_mixtrain=1, dynamic_boa=1, sample_num=8,
               cos_sim_threshold=2e-5, optim_steps=7),
}
N_EXEMPLARS = 256        # synthetic exemplar bank of the retrieval workloads: 10 clusters of ~25 items >= sample_num
W_MB = 107.91            # fp32 parameters (SURVEY.md §8)
FWD_MB = lambda b: 107.91 + 89.51 * b
BWD_MB = lambda b: 215.8 + 133.4 * b


def default_options(**over):
    """Flag defaults of reference dynaboa_benchmark.py:16-65."""
    o = dict(seed=22, seq_seed=22, batch_size=1, lr=3e-6, beta1=0.5, beta2=0.9, use_boa=1, fastlr=8e-6, inner_step=1,
             s2dloss_weight=10.0, shape_prior_weight=2e-6, pose_prior_weight=1e-4, use_frame_losses_lower=1,
             use_frame_losses_upper=1, use_temporal_losses_lower=0, use_temporal_losses_upper=1, sample_num=1, retrieval=1,
             dynamic_boa=1, cos_sim_threshold=3.1e-4, optim_steps=7, lower_level_mixtrain=1, upper_level_mixtrain=1,
             labelloss_weight=0.1, use_meanteacher=1, alpha=0.1, teacherloss_weight=0.1, use_motion=1, interval=5,
             motionloss_weight=0.8, teacher_dropout=1, dataset='3dpw', save_res=0, tensorboard=0, cache_results=0)
    o.update(over)
    return SimpleNamespace(**o)


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (B200_PROFILING.md) through NVML, every 20 ms from a
    thread (the timed region is ~0.15 s: `nvidia-smi -lms` starts too slowly to see it)."""
    REASONS = (('hw_slowdown', 0x8), ('sw_thermal_slowdown', 0x20), ('hw_thermal_slowdown', 0x40), ('sw_power_cap', 0x4))

    def __init__(self, device_index):
        self.sm, self.bits, self.smax, self.h, self.run, self.err = [], 0, None, None, False, None
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            uuid = str(torch.cuda.get_device_properties(device_index).uuid)
            uuid = uuid if uuid.startswith('GPU-') else 'GPU-' + uuid
            try:
                self.h = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByUUID(uuid)
            self.smax = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as e:      # noqa: BLE001
            self.err = f'NVML unavailable: {e}'

    def _sample(self):
        nv = self.nv
        self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
        try:
            self.bits |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
        except Exception:
            self.bits |= int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))

    def _loop(self):
        while self.run:
            try:
                self._sample()
            except Exception as e:      # noqa: BLE001
                self.err = str(e)
                return
            time.sleep(0.02)

    def start(self):
        if self.h is None:
            return
        self.run = True
        self.thread = threading.Thread(target=self._loop, daemon=True)
        self.thread.start()

    def stop(self):
        if self.h is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [self.err or 'NVML unavailable'], 'samples': 0}
        self.run = False
        self.thread.join(timeout=1.0)
        reasons = sorted(name for name, bit in self.REASONS if self.bits & bit)
        return {'sm_mhz': float(np.median(self.sm)) if self.sm else None, 'sm_max_mhz': self.smax, 'reasons': reasons,
                'samples': len(self.sm)}


def load_peaks():
    p = os.path.join(REPO, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
    return 6650.0, 'fallback (B200_PROFILING.md)'


# ------------------------------------------------------------------------------------------------ CPU oracle arm
def build_oracle(workload, n_frames):
    from dynaboa_b200 import constants as C, synthetic
    from oracle import adaptor_ref
    opts = adaptor_ref.default_options(**WORKLOADS[workload])
    gmm = dict(np.load(os.path.join(REPO, 'dynaboa_b200', 'assets', 'gmm_08.npz')))
    bank = synthetic.make_exemplar_bank(n=N_EXEMPLARS) if opts.retrieval else None
    clusters = synthetic.make_clusters(n_items=N_EXEMPLARS) if opts.retrieval else None
    ora = adaptor_ref.OracleAdaptor(opts, synthetic.make_basemodel(),
                                    {g: synthetic.make_smpl_model(g) for g in ('neutral', 'male', 'female')},
                                    synthetic.make_extra_regressors(), gmm, bank=bank, clusters=clusters,
                                    joint_map=C.JOINT_MAP_49, vertex_ids=C.SMPL_EXTRA_VERTEX_IDS, h36m_to_j14=C.H36M_TO_J14)
    return ora, synthetic.SyntheticStream(length=n_frames, batch_size=1)


def pick_threads():
    """Thread count for the CPU arm: the fastest of a few candidates on a short HMR forward+backward probe
    (a 128-thread oneDNN pool on a shared box can be slower than 32 threads)."""
    from dynaboa_b200 import synthetic
    from oracle import hmr_ref
    avail = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
    sd = {k: v.clone().requires_grad_(v.dim() > 0 and 'init_' not in k) for k, v in hmr_ref.strip_prefix(synthetic.make_basemodel()['model']).items()}
    x = torch.randn(1, 3, 224, 224)
    best = (float('inf'), 1)
    for n in sorted({min(c, avail) for c in (8, 16, 32, 64, avail)}):
        torch.set_num_threads(n)
        ts = []
        for _ in range(3):
            t0 = time.perf_counter()
            r, s_, c = hmr_ref.forward(x, sd)
            (r.sum() + s_.sum() + c.sum()).backward()
            ts.append(time.perf_counter() - t0)
        sys.stderr.write(f'[bench] cpu probe: {n} threads -> {min(ts) * 1e3:.0f} ms fwd+bwd\n')
        best = min(best, (min(ts), n))
    torch.set_num_threads(best[1])
    return best[1]


def time_oracle(workload, steps, warmup):
    """Reference CPU path (oracle port), S-adapt scope, best host thread count.  Returns frames/s (median-based)."""
    pick_threads()
    PRELUDE = 7
    warmup = warmup + PRELUDE
    ora, stream = build_oracle(workload, steps + warmup)
    times = []
    for t in range(steps + warmup):
        ora.global_step, ora.fit_losses = t, {}
        t0 = time.perf_counter()
        ora.adaptation(stream[t], with_inference=False)
        ora.predict(stream[t]['image'])
        dt = time.perf_counter() - t0
        sys.stderr.write(f'[bench] cpu frame {t}: {dt:.2f} s\n')
        if t >= warmup:
            times.append(dt)
    return 1.0 / float(np.median(times)), float(np.sum(times))


def time_reference_code(workload, steps, warmup):
    """The reference's OWN CPU implementation (oracle/ref_harness.py: model/hmr.py, base_adaptor.py, dynaboa_benchmark.Adaptor from
    the checkout named by DBOA_REFERENCE_ROOT or the bytecode build() made of it under oracle/_ref, unmodified; smplx / learn2learn restated, synthetic stream), S-adapt scope:
    ``Adaptor.adaptation`` evaluates the model after every inner step and after the outer step (two ``inference`` calls per frame
    in C2), the GPU arm runs ONE output forward per frame -- the time of all but the last ``inference`` call of a frame is
    measured by a wrapper and subtracted.  Returns (frames/s, seconds, description) or None when the reference tree is absent."""
    from dynaboa_b200 import synthetic
    from oracle import ref_harness
    if not ref_harness.available():
        return None
    pick_threads()
    PRELUDE = 7
    warmup = warmup + PRELUDE
    flags = dict(WORKLOADS[workload])
    opts = ref_harness.ref_options(**flags)
    work = tempfile.mkdtemp(prefix='dboa_refarm_')
    n_ex = N_EXEMPLARS if flags['retrieval'] else 64
    synthetic.write_asset_dir(os.path.join(work, 'data'), n_exemplars=n_ex)
    ad = ref_harness.make_reference_adaptor(work, opts, n_exemplars=n_ex)
    stream = synthetic.SyntheticStream(length=steps + warmup, batch_size=1)
    inner = ad.inference
    spent = []

    def timed_inference(*a, **k):
        t0 = time.perf_counter()
        out = inner(*a, **k)
        spent.append(time.perf_counter() - t0)
        return out
    ad.inference = timed_inference
    times = []
    with ref_harness.in_dir(work):
        for t in range(steps + warmup):
            ad.global_step, ad.fit_losses = t, {}
            ad.model.eval()
            del spent[:]
            t0 = time.perf_counter()
            ad.adaptation(stream[t])
            dt = time.perf_counter() - t0 - sum(spent[:-1])
            sys.stderr.write(f'[bench] reference frame {t}: {dt:.2f} s (+ {sum(spent[:-1]):.2f} s of intermediate evaluations, not counted)\n')
            if t >= warmup:
                times.append(dt)
    shutil.rmtree(work, ignore_errors=True)
    root = 'oracle/_ref' if ref_harness.REF == ref_harness.BUILT else ref_harness.REF
    return 1.0 / float(np.median(times)), float(np.sum(times)), f'unmodified reference code from {root} (oracle/ref_harness.py)'


def forward_traffic_mb():
    """DRAM bytes of one dboa_hmr_forward (b=1) from the committed ncu capture; None when the capture is absent."""
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'profiles', 'r02_forward_traffic.json')
    try:
        with open(path) as f:
            d = json.load(f)
        return (d['dram_bytes_read'] + d['dram_bytes_write']) / 1e6
    except (OSError, KeyError, ValueError):
        return None


def cpu_model():
    try:
        for line in open('/proc/cpuinfo'):
            if line.startswith('model name'):
                return line.split(':', 1)[1].strip()
    except Exception:
        pass
    return 'unknown'


def run_reference(args, rank, world):
    if rank != 0:
        return
    ref = time_reference_code(args.workload, args.steps, args.warmup)
    if ref is not None:
        fps, total, how = ref
        kind = 'reference'
    else:
        fps, total = time_oracle(args.workload, args.steps, args.warmup)
        kind, how = 'port', 'oracle/adaptor_ref.py'
    cores = torch.get_num_threads()
    line = {'metric': METRIC, 'value': fps, 'unit': 'frames/s', 'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': 1000.0 / fps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
            'data': 'synthetic', 'impl': 'reference',
            'config': {'workload': f'{args.workload}: 3DPW-shape synthetic stream, S-adapt scope', 'batch': 1,
                       'sample': f'{args.steps} frames on the host CPU'},
            'cpu_baseline': {'value': fps, 'unit': 'frames/s', 'cores': cores, 'kind': kind, 'cpu': cpu_model(),
                             'sample': f'{args.steps} timed frames after {args.warmup} warm-up ({total:.1f} s), {how}'},
            'e2e': {'value': fps, 'unit': 'frames/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}, 'gpu_launches': 0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ GPU arm
def dump_outputs(out_dir, outputs):
    """What the caller of the timed path receives for the last timed frame (rotmat, betas, cam, joints, vertices: ~110 KB), as
    ``<out_dir>/<name>.npy`` in float32, so that two builds can be compared output for output on the same seeded stream."""
    os.makedirs(out_dir, exist_ok=True)
    for name, v in outputs.items():
        np.save(os.path.join(out_dir, f'{name}.npy'), v.detach().float().cpu().numpy())


def run_ours(args, rank, world, local):
    from dynaboa_b200 import _lib, config, dist as ddist, hmr as hmr_mod, synthetic
    from dynaboa_b200.adaptor import Adaptor
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    lib = _lib.load()
    if args.tc >= 0:
        lib.dboa_set_tensor_core_conv(args.tc)
    work = tempfile.mkdtemp(prefix=f'dboa_bench_r{rank}_')
    synthetic.write_asset_dir(os.path.join(work, 'data'), n_exemplars=N_EXEMPLARS if WORKLOADS[args.workload]['retrieval'] else 64)
    config.set_data_root(os.path.join(work, 'data'))
    # untimed frames so that the history ring is full and the motion loss is live (step - interval > 0); with several ranks a few
    # more, so that NCCL's channels and both ranks' allocators are in steady state before the W warm-up steps
    PRELUDE = 7 if world == 1 else 15
    n_frames = PRELUDE + args.steps + args.warmup
    flags = dict(WORKLOADS[args.workload])
    if args.cos_threshold is not None:
        flags['cos_sim_threshold'] = args.cos_threshold
    opts = default_options(expdir=work, expname='bench', model_file=config.BASE_MODEL, synthetic_frames=n_frames, rank=rank, **flags)
    ad = Adaptor(opts)
    ad.fused_eval = 'none'
    if world > 1:
        ddist.attach(ad, world)        # bucketed all-reduce under the upper-level backward, 1/world folded into Adam
    stream = synthetic.SyntheticStream(length=n_frames, batch_size=1, rank=rank)
    keys = ('image', 'smpl_j2d')
    host = [{k: stream[t][k].pin_memory() for k in keys} for t in range(n_frames)]
    resident = [{k: host[t][k].to(dev) for k in keys} for t in range(n_frames)]
    # NSLOT pinned output slots: the outputs of frame t are copied back while the following frames are adapted, and read (event
    # wait) before the slot is reused NSLOT steps later -- every step copies its result to the host inside the timed region.
    # Four slots let the launching thread run up to four frames ahead of the device, so that a host-side hiccup (scheduler,
    # allocator) shorter than a few frames does not drain the device queue.
    NSLOT = 4
    out_host = [{k: torch.empty(s, pin_memory=True) for k, s in (('rotmat', (1, 24, 3, 3)), ('betas', (1, 10)), ('cam', (1, 3)),
                                                                   ('joints', (1, 49, 3)), ('vertices', (1, 6890, 3)))} for _ in range(NSLOT)]
    landed = [None] * NSLOT
    h2d = sum(v.numel() * 4 for v in host[0].values())
    d2h = sum(v.numel() * 4 for v in out_host[0].values())

    def step(t, from_host):
        ad.global_step, ad.fit_losses = t, {}
        if from_host:
            batch = {k: host[t][k].to(dev, non_blocking=True) for k in keys}
        else:
            batch = resident[t]
        ad.adapt(batch)
        if args.serial_output:
            pred = ad.predict(batch['image'])
            if from_host:
                for k, v in out_host[0].items():
                    v.copy_(pred[k], non_blocking=True)
            return pred
        # output forward + SMPL of this frame on the adaptor's side stream: it overlaps the next frame's adaptation
        pred, ev = ad.predict_async(batch['image'])
        if from_host:
            slot = t % NSLOT
            if landed[slot] is not None:
                landed[slot].synchronize()                  # the host has the result that used this slot
            with torch.cuda.stream(ad.output_stream):
                for k, v in out_host[slot].items():
                    v.copy_(pred[k], non_blocking=True)
                landed[slot] = torch.cuda.Event()
                landed[slot].record()
        return pred

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            torch.distributed.barrier()
            torch.cuda.synchronize()

    def timed(from_host):
        ad.reset_records()
        for t in range(PRELUDE + args.warmup):
            step(t, from_host)
        barrier()
        sampler = ClockSampler(local) if rank == 0 and not args.no_clock_sampler else None
        if sampler:
            sampler.start()
        l0 = lib.dboa_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        # no cyclic garbage collection inside the timed region (as timeit does): a full collection walks every object torch has
        # imported (tens of ms) and would stall the launching thread of a 5 ms step
        gc.collect()
        gc.disable()
        try:
            e0.record()
            marks = []
            for t in range(PRELUDE + args.warmup, n_frames):
                pred = step(t, from_host)
                if args.frame_times:                     # diagnostic: one event per frame on the adaptation stream
                    marks.append(torch.cuda.Event(enable_timing=True))
                    marks[-1].record()
            if getattr(ad, 'output_stream', None) is not None:        # the interval ends when the LAST frame's output forward (and its
                torch.cuda.current_stream().wait_stream(ad.output_stream)   # copy-back) on the side stream has finished, not before
            e1.record()
        finally:
            gc.enable()
        barrier()
        ms = e0.elapsed_time(e1)
        if args.frame_times and marks:
            ts = [e0.elapsed_time(m) for m in marks]
            sys.stderr.write('[bench] frame times (ms, adaptation stream): ' + ' '.join(f'{b - a:.2f}' for a, b in zip([0.0] + ts[:-1], ts)) +
                             f' | drain {ms - ts[-1]:.2f}\n')
        launches = lib.dboa_launch_count() - l0
        clocks = sampler.stop() if sampler else None
        return ddist.max_over_ranks(ms, dev), launches, clocks, pred

    # reset model state between the two measurements so both see the same trajectory
    snapshot = (ad.model.module.arena.clone(), ad.teacher.arena.clone())

    def restore():
        ad.model.module.arena.copy_(snapshot[0]); ad.teacher.arena.copy_(snapshot[1])
        ad.optimizer.m.zero_(); ad.optimizer.v.zero_(); ad.optimizer.step_count = 0

    sys.stderr.write('[bench] setup done\n')
    ms_dev, launches, clocks, last = timed(False)
    sys.stderr.write(f'[bench] device-resident: {ms_dev / args.steps:.2f} ms/frame\n')
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)
    restore()
    ms_e2e, _, clocks_e2e, _ = timed(True)
    value = world * args.steps / (ms_dev / 1000.0)
    e2e = world * args.steps / (ms_e2e / 1000.0)

    # ---- roofline of the dominant unit: the HMR forward launch sequence (b = 1), timed alone with CUDA events
    roof = None
    cpu_base = None
    if rank == 0:
        peak, peak_src = load_peaks()
        model = ad.model.module
        x = resident[0]['image']
        tape = torch.empty(hmr_mod.tape_floats(1), dtype=torch.float32, device=dev)
        flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
        for _ in range(3):
            hmr_mod.raw_forward(model.arena, model._buffers, x, None, tape)
        torch.cuda.synchronize()
        reps, tot = 20, 0.0
        l0 = lib.dboa_launch_count()
        for _ in range(reps):
            flush.zero_()                                            # evict L2 (126 MB) between timed iterations
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            hmr_mod.raw_forward(model.arena, model._buffers, x, None, tape)
            b.record()
            torch.cuda.synchronize()
            tot += a.elapsed_time(b)
        fwd_ms = tot / reps
        fwd_launches = (lib.dboa_launch_count() - l0) // reps
        achieved = FWD_MB(1) / 1e3 / (fwd_ms / 1e3)
        roof = {'bound': 'hbm', 'kernel': f'dboa_hmr_forward b=1 ({fwd_launches} launches: fused plan -- stride-1 convs apply the GroupNorm of their operand on load)',
                'achieved': achieved, 'peak': peak, 'peak_source': peak_src, 'unit': 'GB/s', 'frac': achieved / peak,
                'traffic': forward_traffic_mb(), 'traffic_unit': 'MB per forward (dram__bytes_read.sum + dram__bytes_write.sum, ncu capture '
                'profiles/r02_forward_traffic.json)', 'algorithmic_MB_per_launch': FWD_MB(1), 'ms_per_launch': fwd_ms,
                'step_model': {'algorithmic_GB_per_frame': 3.63, 'achieved_GBps': 3.63 / (ms_dev / 1000.0 / args.steps),
                               'frac': 3.63 / (ms_dev / 1000.0 / args.steps) / peak}}
        if world == 1 and not args.no_cpu_baseline:
            ref = time_reference_code(args.workload, args.cpu_frames, 1)
            if ref is not None:
                fps, total, how = ref
                kind = 'reference'
            else:
                fps, total = time_oracle(args.workload, args.cpu_frames, 1)
                kind, how = 'port', 'oracle/adaptor_ref.py'
            cpu_base = {'value': fps, 'unit': 'frames/s', 'cores': torch.get_num_threads(), 'kind': kind, 'cpu': cpu_model(),
                        'sample': f'{args.cpu_frames} frames of the same stream after 1 warm-up ({total:.1f} s), {how}'}
        line = {'metric': METRIC, 'value': value, 'unit': 'frames/s', 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
                'ms_per_step': ms_dev / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
                'data': 'synthetic',
                'config': {'workload': f'{args.workload}: 3DPW-shape synthetic stream, batch 1 per GPU, S-adapt scope '
                                       '(adaptation + one output forward/SMPL)', 'flags': flags,
                           'output': 'serial' if args.serial_output else 'output forward + SMPL of frame t on a side stream, overlapped with '
                           'the adaptation of frame t+1 (same weights; the optimiser step waits for the read); --serial-output disables',
                           'parallelism': f'dp{world}: frames sharded over ranks, the 107.9 MB outer gradient all-reduced in 3 buckets '
                           'under the upper-level backward (NCCL on a communication stream), 1/world folded into Adam'
                           if world > 1 else 'single GPU',
                           'dynamic_steps': (list(ad.optim_step_record[-args.steps:]) if WORKLOADS[args.workload]['dynamic_boa'] else None),
                           'one_minus_cos12_first_test': ([round(1.0 - v[0][12]['cos'], 7) for _, v in sorted(ad.feat_sims.items())][-args.steps:]
                                                          if WORKLOADS[args.workload]['dynamic_boa'] else None),
                           'l2': 'per-step working set (theta, fast weights, Adam m/v, teacher, gradient arena: 6 x 108 MB + '
                                 'activations) exceeds the 126 MB L2; the isolated forward timing flushes L2 with a 256 MB memset'},
                'e2e': {'value': e2e, 'unit': 'frames/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
                        'ms_per_step': ms_e2e / args.steps},
                'gpu_launches': int(launches), 'clocks': clocks, 'roofline': roof, 'cpu_baseline': cpu_base}
        print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='c2', choices=sorted(WORKLOADS))
    ap.add_argument('--cpu-frames', type=int, default=8)
    ap.add_argument('--cos-threshold', type=float, default=None,
                    help='override cos_sim_threshold of a dynamic_boa workload (the reference default 3.1e-4 never fires on the synthetic stream)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--frame-times', action='store_true', help='diagnostic: per-frame times of the timed region on stderr')
    ap.add_argument('--no-clock-sampler', action='store_true', help='diagnostic: no NVML polling during the timed region')
    ap.add_argument('--serial-output', action='store_true',
                    help='run the output forward on the adaptation stream (no overlap with the next frame)')
    ap.add_argument('--tc', type=int, default=-1, help='tensor-core conv mode override (0 fp32 CUDA cores, 1 forward, 2 forward+dgrad+wgrad, 3 forward+dgrad)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write the outputs of the last timed frame as DIR/<name>.npy (rank 0)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs applies to the GPU path (--impl ours)')
    if args.warmup < 3 and args.impl == 'ours':
        args.warmup = 3
    from dynaboa_b200 import dist as ddist
    if args.impl == 'reference':
        rank = int(os.environ.get('RANK', '0'))
        run_reference(args, rank, int(os.environ.get('WORLD_SIZE', '1')))
        return
    rank, world, local = ddist.init_from_env()
    if world != args.gpus and world > 1:
        raise SystemExit(f'--gpus {args.gpus} but WORLD_SIZE={world}')
    run_ours(args, rank, world, local)
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == '__main__':
    main()
