#!/usr/bin/env python
"""bench.py -- lnlike evals/sec of the batched likelihood hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

`--dump-outputs DIR` writes the lnL vector of the last timed step as DIR/lnl.npy (float64).  Every input
(networks, mock observation, live points) comes from fixed seeds and the CPU oracle, never from the build
being measured, so two builds run with the same arguments can be compared file by file.

One "step" = one pass of the whole hot path (emulator MLP -> broadening tail -> chi2) over a
batch of B synthetic live points of config C2 (SURVEY.md §8d: LinNet 4-256-256-256-14172,
UVES-range mock, n_obs 7000).  N>1: one process per GPU (torchrun), B points per GPU (weak
scaling), replicated weights, one NCCL all-gather of the lnL vector per step.

`--impl reference` times the reference's own likelihood path on all host cores: the UNMODIFIED
reference files staged under oracle/_ref (oracle/make_ref.py copies them byte for byte in the build
container; the directory is git-ignored and ships with the gpurun snapshot), driven through
oracle/refharness.py exactly as the golden fixtures were minted -- kind "reference".  Only when that
directory is absent does the arm fall back to the oracle port (kind "port").  Same workload string,
same theta seed and the same points per step as the CUDA arm.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = 'lnlike_evals_per_sec'
UNIT = 'evals/s'


def load_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return d['hbm_gbs'], d['bf16_tflops'], d.get('bf16_tflops_sustained', d['bf16_tflops']), 'measured'
    return 6650.0, 1590.0, 1400.0, 'fallback'


# --------------------------------------------------------------------------- CPU baseline
_W = {}


def reference_kind():
    """'reference' when the unmodified reference files are present (oracle/_ref or /root/reference)."""
    from oracle import refharness
    return 'reference' if refharness.available() else 'port'


def make_cpu_like(cfg, kind, vector_chi2=False):
    """Scalar ``lnlikefn(theta_row) -> float`` of the reference (or of the oracle port)."""
    if kind == 'reference':
        import warnings
        warnings.filterwarnings('ignore')
        from oracle import refharness
        like = refharness.build_likelihood(cfg)
        if vector_chi2:
            refharness.vectorise_chi2(like)
        return like.lnlikefn
    from oracle import payne_oracle as O
    return O.OracleLikelihood(cfg).lnlikefn


def _cpu_init(cfg, kind, threads):
    import torch
    assert not torch.cuda.is_available(), 'the CPU arm must not see a GPU (the reference would move its net there)'
    if threads:
        torch.set_num_threads(threads)
    _W['fn'] = make_cpu_like(cfg, kind)


def _cpu_eval(rows):
    fn = _W['fn']
    return [float(fn(r)) for r in rows]


def _cpu_rate(args):
    """(seconds, vector_chi2) -> (evals/s, points) of one process looping lnlikefn over its rows."""
    rows, seconds, vector, cfg, kind = args
    fn = make_cpu_like(cfg, kind, vector_chi2=True) if vector else _W['fn']
    for r in rows[:3]:
        fn(r)
    n, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < seconds and n < len(rows):
        fn(rows[n])
        n += 1
    return n / (time.perf_counter() - t0), n


class CpuPool:
    """Host-core worker processes, one likelihood object each (the reference evaluates one parameter
    vector per call).  The workers are spawned with CUDA hidden: on a GPU host the reference's
    ``predictspec.py:16-20`` would otherwise put its tensors on the device, and this arm times the
    reference's CPU path."""

    def __init__(self, cfg, cores=None, kind='reference', threads=1):
        import multiprocessing as mp
        self.cores = cores or os.cpu_count() or 1
        self.kind = kind
        keep = os.environ.get('CUDA_VISIBLE_DEVICES')
        os.environ['CUDA_VISIBLE_DEVICES'] = ''
        try:
            self.pool = mp.get_context('spawn').Pool(self.cores, initializer=_cpu_init, initargs=(cfg, kind, threads))
            self.pool.map(_cpu_eval, [[] for _ in range(self.cores)])      # workers are up (env captured)
        finally:
            if keep is None:
                del os.environ['CUDA_VISIBLE_DEVICES']
            else:
                os.environ['CUDA_VISIBLE_DEVICES'] = keep

    def run(self, theta):
        chunks = [c for c in np.array_split(theta, self.cores * 2) if len(c)]
        t0 = time.perf_counter()
        out = self.pool.map(_cpu_eval, chunks)
        dt = time.perf_counter() - t0
        return np.concatenate([np.asarray(o) for o in out]), dt

    def close(self):
        self.pool.close()
        self.pool.join()


def single_process_lines(cfg, theta, kind, seconds=4.0):
    """SURVEY §8d / BASELINE.md §3: one process with 1 thread, one process with torch's default thread
    count, and the vectorised-chi2 variant (likelihood.py:95-97 is a Python generator, ~40 % of the
    reference).  Each runs in its own CUDA-blind worker process."""
    out = {}
    rows = np.ascontiguousarray(theta[:512])
    for key, threads, vector in [('one_process_1_thread', 1, False), ('one_process_default_threads', None, False),
                                 ('one_process_1_thread_vectorised_chi2', 1, True)]:
        if vector and kind != 'reference':
            continue
        pool = CpuPool(cfg, 1, kind, threads)
        v, n = pool.pool.apply(_cpu_rate, ((rows, seconds, vector, cfg, kind),))
        pool.close()
        out[key] = {'value': v, 'unit': UNIT, 'points': n}
    return out


# --------------------------------------------------------------------------- clocks
class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.sm, self.reasons, self.max_sm = index, False, [], set(), None
        # NVML polling is not free for the polled GPU's process: at 8 GPUs a 2 ms period measured +7 us per 0.87 ms step
        # against a 50 ms period (gpurun_out/r2_bench_n8c.json); 4 ms still gives 4-5 samples in the shortest runs
        self.period = float(os.environ.get('BENCH_CLOCK_PERIOD', '0.004'))
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: 'hw_slowdown',
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: 'hw_thermal_slowdown',
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: 'sw_thermal_slowdown',
                 nv.nvmlClocksThrottleReasonSwPowerCap: 'sw_power_cap'}
        while not self.stop_flag:
            try:
                self.sm.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(self.period)

    def summary(self):
        return {'sm_mhz': float(np.median(self.sm)) if self.sm else None, 'sm_max_mhz': self.max_sm,
                'reasons': sorted(self.reasons), 'samples': len(self.sm)}


# --------------------------------------------------------------------------- config
def build_c2():
    """C2 with the mock observation from the CPU oracle: the inputs do not depend on the build being measured."""
    from oracle import payne_oracle as O
    from thepayne_b200 import synth
    return synth.config_c2(O.model_fn)


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(path, arrays):
    """Write every array as <path>/<name>.npy in float64, DUMP_MAX_BYTES at most in all.  An array over its share is
    replaced by a fixed sample of its elements (seed 0, in index order): the same positions for every run of the
    same shape."""
    os.makedirs(path, exist_ok=True)
    keep = DUMP_MAX_BYTES // max(1, len(arrays)) // 8
    for name, a in arrays.items():
        a = np.asarray(a, dtype=np.float64)
        if a.size > keep:
            a = a.ravel()[np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))]
        np.save(os.path.join(path, name + '.npy'), a)


def bench_config(B, D_out, n_obs):
    """The `config` object both arms print (so the driver sees the same workload on both)."""
    return {'workload': 'C2-uves: LinNet 4-256-256-256-%d random-init, n_obs %d, FFT 16384, theta seed 1234' % (D_out, n_obs),
            'points_per_gpu': B,
            'l2': 'per-step working set (flux slab %.0f MB) exceeds the 126 MB L2; no explicit flush'
                  % (B * D_out * 4 / 1e6)}


def other_configs(precision):
    """Device-resident throughput of the other BASELINE.json configs on one GPU (few steps each)."""
    import torch
    from thepayne_b200 import synth
    from thepayne_b200.engine import engine_from_config
    out = {}

    def gpu_model_fn(cfg, theta):
        n = len(cfg.obs_wave)
        cfg.obs_flux, cfg.obs_eflux = np.ones(n), np.ones(n)
        if cfg.phot is not None:
            cfg.obs_phot = {b: [0.0, 1.0] for b in cfg.phot.bands}
        eng = engine_from_config(cfg, precision=precision)
        fl, mg, _ = eng.model_batch(torch.from_numpy(np.ascontiguousarray(theta)).cuda())
        r = (fl.cpu().numpy(), None if mg is None else mg.cpu().numpy())
        eng.close()
        return r
    for key, builder, B, steps, what in [
            ('c3_joint', synth.config_c3, 16384, 5, 'C3: C2 + 7-band photometry (SED nets H=128), 16384 points'),
            ('c4_monolithic', synth.config_c4, 4096, 3,
             'C4 (i): LinNet 5-512-512-512-51784, 65536-sample transforms (one per cluster of four CTAs), n_obs 25000, '
             'order-4 continuum, Vrot<=100; 4096-point slabs of the 64k-point batch')]:
        try:
            cfg = builder(gpu_model_fn)
            eng = engine_from_config(cfg, precision=precision)
            eng.set('max_batch', 8192 if key == 'c3_joint' else 4096)
            th = torch.from_numpy(np.ascontiguousarray(cfg.draw(B, seed=99))).cuda()
            for _ in range(2):
                o = eng.lnlike_batch(th)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                o = eng.lnlike_batch(th)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            out[key] = {'workload': what, 'points': B, 'ms_per_step': ms, 'value': B / (ms * 1e-3), 'unit': UNIT,
                        'finite_lnl': int(torch.isfinite(o).sum().item())}
            if key == 'c4_monolithic':
                out[key]['tail_cluster'] = int(eng.query('tail_cluster'))
            eng.close()
            del th, o
            torch.cuda.empty_cache()
        except Exception as e:                      # an extra line must never cost the headline
            out[key] = {'error': str(e)[:200]}
    return out


def mlp_flops(cfg):
    dims = [w.shape for w in cfg.spec.weights]
    return 2.0 * sum(o * i for o, i in dims)


# --------------------------------------------------------------------------- arms
def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    kind = reference_kind()
    cfg = build_c2()
    cores = os.cpu_count() or 1
    pool = CpuPool(cfg, cores, kind)
    B = args.batch
    theta = cfg.draw(B, seed=1234)                 # the CUDA arm's rank-0 batch
    # Bound the run: a step is the first S points of the B-point batch, S = B when the whole
    # --steps/--warmup run then stays within ~4 minutes on this host, else the largest multiple of
    # the core count that does (probe: one round of 4 points per core).
    pool.run(theta[:cores])
    _, dt = pool.run(theta[:4 * cores])
    per_point = dt / (4 * cores)
    nsteps = args.steps + args.warmup
    S = B
    if per_point * B * nsteps > 240.0:
        S = max(cores, int(240.0 / (per_point * nsteps)) // cores * cores)
    for i in range(args.warmup):
        pool.run(theta[:S])
    tot = 0.0
    for i in range(args.steps):
        lnl, dt = pool.run(theta[:S])
        tot += dt
    pool.close()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {'lnl': lnl})
    v = S * args.steps / tot
    sample = ('%d of the %d points per step x %d steps, scalar lnlikefn per point, %d procs x 1 thread; '
              'implementation: %s' % (S, B, args.steps, cores,
                                      'unmodified reference files (oracle/_ref)' if kind == 'reference' else 'oracle port'))
    print(json.dumps({
        'impl': 'reference', 'metric': METRIC, 'value': v, 'unit': UNIT, 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * tot / args.steps * (B / S),
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'fp32 MLP / fp64 tail',
        'data': 'synthetic', 'config': bench_config(B, cfg.spec.D_out, len(cfg.obs_wave)),
        'cpu_baseline': {'value': v, 'unit': UNIT, 'cores': cores, 'kind': kind, 'sample': sample},
        'e2e': {'value': v, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0}))


def run_ours(args):
    import torch
    import torch.distributed as dist
    from thepayne_b200 import dist as pdist
    from thepayne_b200.engine import engine_from_config

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    B, K, W = args.batch, args.steps, args.warmup
    cfg = build_c2()
    # A throw-away engine evaluates the truth once before the timed engine is made.  Without it the timed engine, then
    # the first on the device, ran 0.2 % slower per step (one B200 at 1000 W: 0.8551 against 0.8534 ms, alternated runs).
    warm = engine_from_config(cfg, precision=args.precision)
    warm.model_batch(torch.from_numpy(np.ascontiguousarray(cfg.theta_true[None, :])).cuda())
    warm.close()
    eng = engine_from_config(cfg, precision=args.precision)
    eng.set('max_batch', args.slab)
    theta_h = np.ascontiguousarray(cfg.draw(B, seed=1234 + rank))    # rank 0: the reference arm's batch
    theta = torch.from_numpy(theta_h).cuda()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # N > 1: the all-gather of step i runs on a side stream beside the kernels of step i + 1
    # (thepayne_b200.dist.PipelinedGather); the timed region ends only after the last gather has landed
    # N > 1: the library's own all-gather fused into the tail kernel (payne_lnlike_batch_gather: the thread that writes a
    # point's lnL stores it into every peer's buffer over NVLink, the last CTA raises the flags).  Measured on one 8 x B200
    # box, same run: 0.8626 ms/step against 0.8729 with ncclAllGather on a side stream one step behind
    # (BENCH_GATHER=nccl, the fallback when peer memory cannot be mapped); 0.853-0.857 per rank without any gather.
    pg = pdist.PipelinedGather() if world > 1 else None
    gather_kind = 'ncclAllGather on a side stream, one step behind (dist.PipelinedGather)' if world > 1 else None
    peer_main = None
    if world > 1 and os.environ.get('BENCH_GATHER', 'peer') == 'peer':
        try:
            peer_main = pdist.PeerGather(eng, B)
            gather_kind = 'peer memory, fused into the tail kernel (dist.PeerGather)'
        except Exception:
            peer_main = None

    def step():
        if peer_main is not None:
            return peer_main.submit(theta)
        lnl = eng.lnlike_batch(theta)
        if world == 1:
            return lnl
        return pg.submit(lnl)

    def drain():
        if peer_main is not None:
            return peer_main.flush()
        return pg.flush()[-1] if world > 1 else None

    for _ in range(max(W, 3)):
        out = step()
    if world > 1:
        out = drain()
    barrier()
    # N > 1: the same K steps WITHOUT the gather first -- every rank at its own pace.  With the gather the ranks are
    # coupled (all run at the pace of the slowest GPU of the box); the uncoupled times tell that apart from a cost of
    # the collective (by_rank in the line).
    ms_free = None
    if world > 1:
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        for _ in range(K):
            eng.lnlike_batch(theta)
        f1.record()
        barrier()
        ms_free = f0.elapsed_time(f1)
    sampler = ClockSampler(local)
    sampler.start()
    l0 = eng.query('launches')
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(K):
        out = step()
    if world > 1:
        out = drain()                     # the compute stream waits for the last gather
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = eng.query('launches') - l0
    sampler.stop_flag = True
    sampler.join()
    by_rank = None
    if world > 1:
        # the step time is the MAX over ranks; every rank's own time and SM clock go into the line as well, so that a
        # scaling loss can be told apart from one slow GPU of the box
        mine = torch.tensor([ms, float(np.median(sampler.sm)) if sampler.sm else 0.0, ms_free], device='cuda', dtype=torch.float64)
        allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        by_rank = {'ms_per_step': [round(float(a[0].item()) / K, 5) for a in allr],
                   'ms_per_step_without_gather': [round(float(a[2].item()) / K, 5) for a in allr],
                   'sm_mhz': [float(a[1].item()) for a in allr]}
        ms = max(float(a[0].item()) for a in allr)
    n_finite = int(torch.isfinite(out).sum().item())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {'lnl': out.cpu().numpy()})

    # per-kernel device time (CUDA events on the launching stream inside the library)
    eng.set('timing', 1)
    mlp_ms = tail_ms = 0.0
    for _ in range(K):
        eng.lnlike_batch(theta)
        tail_ms += eng.last_ms('tail')
        mlp_ms += eng.last_ms('mlp')
    eng.set('timing', 0)
    mlp_ms /= K
    tail_ms /= K

    # end to end: host theta in, host lnL out, every step.  N = 1: the host-buffer C-ABI entry
    # (pinned staging + H2D + kernels + D2H inside the library).  N > 1: pinned theta -> H2D -> kernels ->
    # NCCL all-gather of lnL -> D2H of the gathered vector, i.e. what a sampler on every rank would see.
    if world == 1:
        def e2e_step():
            return eng.lnlike_batch(theta_h)
    else:
        theta_pin = torch.from_numpy(theta_h).pin_memory()
        lnl_pin = torch.empty(world * B, dtype=torch.float64).pin_memory()
        # every step needs ITS gathered vector (nothing to pipeline behind): the library's own all-gather over peer
        # memory (payne_gather_*: one push kernel + flags, ~13 us at 8 GPUs) instead of a blocking ncclAllGather
        try:
            peer = peer_main if peer_main is not None else pdist.PeerGather(eng, B)
            e2e_gather = 'peer memory (payne_lnlike_batch_gather + payne_gather_flush)'
        except Exception as exc:                     # raised on every rank alike
            peer, e2e_gather = None, 'ncclAllGather (peer memory unavailable: %s)' % str(exc)[:80]

        def e2e_step():
            th = theta_pin.cuda(non_blocking=True)
            if peer is not None:
                peer.submit(th)
                g = peer.flush()
            else:
                g = pdist.gather_equal(eng.lnlike_batch(th))
            lnl_pin.copy_(g, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            return lnl_pin.numpy()
    for _ in range(2):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(K):
        lnl_h = e2e_step()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], device='cuda')
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())

    # C5 (BASELINE config 5): a 2^20-point sweep of the same workload split over the N GPUs (strong
    # scaling: total work fixed), slabs of 8192 points, one all-gather of the full lnL vector per step
    c5 = None
    if not args.no_extra:
        total = 1 << 20
        per = total // world
        th5 = torch.from_numpy(np.ascontiguousarray(cfg.draw(per, seed=777 + rank))).cuda()
        eng.set('max_batch', 8192)

        def step5():
            lnl = eng.lnlike_batch(th5)
            return pdist.gather_equal(lnl) if world > 1 else lnl
        step5()
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        for _ in range(3):
            o5 = step5()
        f1.record()
        barrier()
        ms5 = f0.elapsed_time(f1)
        if world > 1:
            t = torch.tensor([ms5], device='cuda')
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms5 = float(t.item())
        c5 = {'workload': 'C5: 2^20-point sweep of the C2 workload, strong scaling', 'points_total': per * world,
              'points_per_gpu': per, 'value': per * world * 3 / (ms5 * 1e-3), 'unit': UNIT, 'ms_per_step': ms5 / 3,
              'finite_lnl': int(torch.isfinite(o5).sum().item())}
        del th5, o5
        eng.set('max_batch', args.slab)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    hbm, tf_burst, tf_sust, which = load_peaks()
    D_out, n_obs = cfg.spec.D_out, len(cfg.obs_wave)
    tail_bytes = B * (4.0 * D_out + 4.0)                 # SURVEY §8d: read the fp32 flux row once + lnL
    traffic, limiter = None, None
    try:
        tfile = json.load(open(os.path.join(ROOT, 'profiles', 'roofline_traffic.json')))
        tj = tfile['tail']
        if tj['points'] == B:
            traffic = tj['dram_bytes']
        limiter = tfile.get('tail_limiter')
    except Exception:
        pass
    tail_gbs = tail_bytes / (tail_ms * 1e-3) / 1e9
    # the two on-chip rooflines the tail actually runs against (VERDICT r1 1e): shared-memory wavefronts
    # (128 B per clock per SM) and warp-instruction issue (4 per clock per SM), per-point counts from the
    # committed ncu census, live time and live SM clock
    smem_roof = issue_roof = None
    try:
        cen = tfile['tail_census']
        clk = (sampler.summary().get('sm_mhz') or sampler.summary().get('sm_max_mhz') or 1965.0) * 1e6
        sms = eng.query('sm_count')
        wf, wfi, wi = cen['smem_wavefronts_per_point'], cen['smem_wavefronts_ideal_per_point'], cen['warp_instructions_per_point']
        a = wfi * 128.0 * B / (tail_ms * 1e-3) / 1e9
        pk = sms * 128.0 * clk / 1e9
        smem_roof = {'kernel': 'tail_fast_kernel', 'bound': 'shared-memory', 'achieved': a, 'peak': pk, 'unit': 'GB/s',
                     'frac': a / pk, 'frac_with_conflict_replays': wf * 128.0 * B / (tail_ms * 1e-3) / 1e9 / pk,
                     'wavefronts_per_point': wf, 'ideal_wavefronts_per_point': wfi,
                     'note': 'conflict-free wavefronts x 128 B per point x points / live tail time, against SMs x 128 B/clk x '
                             'live SM clock; counts from ' + cen['source']}
        ai = wi * B / (tail_ms * 1e-3) / 1e9
        pi = sms * 4.0 * clk / 1e9
        issue_roof = {'kernel': 'tail_fast_kernel', 'bound': 'issue', 'achieved': ai, 'peak': pi, 'unit': 'G warp-inst/s',
                      'frac': ai / pi, 'warp_instructions_per_point': wi,
                      'note': 'executed warp instructions per point x points / live tail time, against SMs x 4 schedulers x '
                              'live SM clock; the kernel is co-limited by issue and the shared-memory pipe (DESIGN.md 3.3)'}
    except Exception:
        pass
    fl = mlp_flops(cfg) * B
    mlp_tfs = fl / (mlp_ms * 1e-3) / 1e12
    res = {
        'metric': METRIC, 'value': world * B * K / (ms * 1e-3), 'unit': UNIT, 'n_gpus': world, 'steps': K,
        'warmup': max(W, 3), 'ms_per_step': ms / K, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'fp32 (tcgen05 bf16x3 exact-accumulation MLP, fp32 FFT tail, fp64 chi2)'
        if args.precision == 'parity' else args.precision,
        'data': 'synthetic',
        'config': bench_config(B, D_out, n_obs), 'precision_mode': args.precision, 'finite_lnl': n_finite,
        'clocks': sampler.summary(),
        'e2e': {'value': world * B * K / e2e_s, 'unit': UNIT, 'h2d_bytes_per_step': int(theta_h.nbytes),
                'd2h_bytes_per_step': int(lnl_h.nbytes),
                'path': 'payne_lnlike_batch_host (C ABI, host buffers)' if world == 1 else
                        'pinned theta -> H2D -> likelihood -> all-gather of lnL over %s -> D2H' % e2e_gather},
        'gpu_launches': int(launches),
        'by_rank': by_rank, 'gather': gather_kind,
        'roofline': {'kernel': 'tail_fast_kernel<%d> (+tail_setup_kernel)' % int(np.log2(eng.query('nfft1'))), 'bound': 'hbm', 'achieved': tail_gbs, 'peak': hbm, 'unit': 'GB/s',
                     'frac': tail_gbs / hbm, 'traffic': traffic, 'algorithmic_bytes': tail_bytes, 'peak_source': which, 'ms_per_launch': tail_ms,
                     'limiter': limiter,
                     'note': 'algorithmic bytes = B*(4*D_out+4). The kernel cannot be HBM-bound under reference '
                             'semantics: 4 in-shared-memory FFTs of 16384 samples per point make the L1/shared-memory '
                             'data pipe the busiest unit (limiter, from the committed ncu capture); see DESIGN.md'},
        'roofline_smem': smem_roof, 'roofline_issue': issue_roof,
        'roofline_mlp': {'kernel': 'tc_gemm_kernel x5 (+lin1)', 'bound': 'tensor', 'achieved': mlp_tfs,
                         'peak': tf_burst / 2, 'unit': 'TFLOP/s', 'frac': mlp_tfs / (tf_burst / 2),
                         'ms_per_step': mlp_ms,
                         'issued_bf16_tflops': 6 * mlp_tfs if args.precision == 'parity' else None,
                         'issued_frac_of_bf16_peak': 6 * mlp_tfs / tf_burst if args.precision == 'parity' else None,
                         'note': 'algorithmic flops (one MMA per product) vs TF32-equivalent peak = measured '
                                 'bf16 burst / 2 (%s); parity mode issues 6 bf16 MMAs per product, so the tensor pipe '
                                 'sees issued_bf16_tflops against the bf16 burst peak; ms_per_step also holds the '
                                 'encode kernel and four latency-bound 256x256 hidden layers' % which},
    }
    if world == 1 and not args.no_cpu:
        cores = os.cpu_count() or 1
        kind = reference_kind()
        pool = CpuPool(cfg, cores, kind)
        S = max(64, 8 * cores)
        pool.run(theta_h[:min(S, B)])          # warm-up (spawn + first torch call)
        n, tot, dl = 0, 0.0, 0.0
        lnl_gpu = out[:B].cpu().numpy()
        i = 0
        while tot < args.cpu_seconds and (i + 1) * S <= B:
            r, dt = pool.run(theta_h[i * S:(i + 1) * S])
            dl = max(dl, float(np.nanmax(np.abs(r - lnl_gpu[i * S:(i + 1) * S]))))
            tot += dt
            n += S
            i += 1
        pool.close()
        res['cpu_baseline'] = {'value': n / tot, 'unit': UNIT, 'cores': cores, 'kind': kind,
                               'per_core': n / tot / cores,
                               'sample': '%d of the %d timed points, scalar lnlikefn per point, %d procs x 1 thread; %s'
                                         % (n, B, cores, 'unmodified reference files (oracle/_ref)' if kind == 'reference'
                                            else 'oracle port'),
                               'max_abs_dlnl_vs_gpu': dl}
        res['cpu_baseline'].update(single_process_lines(cfg, theta_h, kind, seconds=min(4.0, args.cpu_seconds / 3)))
    if c5 is not None:
        res['c5_sweep'] = c5
    if world == 1 and not args.no_extra:
        eng.close()
        res['other_configs'] = other_configs(args.precision)
    print(json.dumps(res))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=100)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--batch', type=int, default=4096)
    ap.add_argument('--slab', type=int, default=8192)
    ap.add_argument('--precision', default='parity')
    ap.add_argument('--cpu-seconds', type=float, default=12.0)
    ap.add_argument('--no-cpu', action='store_true')
    ap.add_argument('--no-extra', action='store_true', help='skip the C3/C4/C5 extra lines')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the lnL of the last timed step to DIR/lnl.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
