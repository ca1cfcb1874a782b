#!/usr/bin/env python
"""bench.py -- chunks/s and real-time factor of the full encode -> stage 1 -> stage 2 -> vocode path.

  python bench.py --gpus 1 --steps K --warmup W            (driver; N > 1 via torch.distributed.run)
  python bench.py --impl reference ...                      (the CPU implementation of the same path)

A "step" is one 0.3 s @ 24 kHz chunk of one audio stream pushed through the device-resident session
(BASELINE.json configs[1]: single stream, buffer_time = 0.3 s, extras (0, 0.5, 0), frame 5 ms;
stage-1 / stage-2 U-Nets at base width 64 with seeded synthetic weights; synthetic speech).
  value : chunks/s with the chunk's samples already in HBM and the output left there
          (ryk_session_push_device), K consecutive chunks, CUDA events, max over ranks
  e2e   : the same K chunks through ryk_session_push with HOST buffers (H2D + kernels + D2H per step)
Multi-GPU: one independent stream per rank ("weak"); NCCL only broadcasts the weights at init.
"""
import argparse
import json
import os
import sys

# before anything creates the CUDA context: a session drives 7 streams, a group of 8 sessions 57 (see ryk_engine_create)
os.environ.setdefault('CUDA_DEVICE_MAX_CONNECTIONS', '32')
import tempfile
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

BUFFER_TIME = 0.3
EXTRA = (0.0, 0.5, 0.0)
FS = 24000
THRESHOLD_DB = 60.0
METRIC = 'chunks_per_s_0.3s_24kHz_encode_stage1_stage2_vocode'
DUMP_BYTES = 64 << 20          # --dump-outputs: at most this much in all, over every rank and stream
WORKLOAD = ('single stream per GPU, buffer_time=0.3 s, extras (0,0.5,0), frame_period 5 ms, 24 kHz in/out, '
            'convert window 260 -> 384 frames, stage-1 1-D U-Net base 64 (13.6 M params), '
            'stage-2 2-D U-Net base 64 on 384x512 (54.4 M params, 142 GFLOP/chunk), WORLD DIO+StoneMask/CheapTrick/D4C + realtime synthesis')


# algorithmic work of the stage-2 k4 layers (the tcgen05 kernel launches) for one 384x512 forward, base 64
STAGE2_TC_FLOP = None


def stage2_tc_flop(Tp=384, base=64):
    enc = [1, 2, 4, 8, 8, 8, 8, 8]
    dec = [8, 8, 8, 8, 4, 2, 1]
    fl = 0.0
    for i in range(1, 8):
        cin, cout = base * enc[i - 1], base * enc[i]
        fl += 2.0 * 16 * cin * cout * (Tp >> i) * (512 >> i)
    for d in range(7):
        cin = base * enc[7] if d == 0 else base * dec[d - 1] + base * enc[7 - d]
        cout = base * dec[d]
        fl += 2.0 * 16 * cin * cout * (Tp >> (7 - d)) * (512 >> (7 - d))
    return fl


# short device-resident legs of BASELINE configs 3 and 5 plus 4 grouped streams of the headline chunk size (buffer_time, streams per GPU, steps)
EXTRA_LEGS = ((0.1, 1, 20), (1.0, 1, 12), (1.0, 8, 8), (0.3, 4, 12))

DTYPE = ('f64 (WORLD analysis / synthesis, SPTK), f16 operands / f32 accumulate: stage-2 k4 layers on tcgen05, stage-1 k4 layers on mma.sync '
         'inside the one-launch cluster kernel; f32 CUDA cores (3x3 / k3 edge layers)')


def bench_config(workload, B=1):
    """`config` of the JSON line -- built by ONE function so that the repo arm and the reference arm carry identical keys."""
    return dict(
        workload=workload,
        timing='CUDA events on the engine stream (forked to / joined from the session streams) around the K pushes, max over ranks',
        pipeline='gate | analysis (2 chunks in flight) | stage 1 | stage 2 | synthesis of consecutive chunks overlap on 6 CUDA streams per audio '
                 'stream, each stage a CUDA graph (the reference overlaps its 3 worker processes); e2e keeps 4 steps in flight',
        l2='per-step footprint (109 MB fp16 stage-2 weights + 54 MB stage-1 weights + ~100 MB activations) exceeds the 126 MB L2; no explicit flush',
        streams_per_gpu=B, silence_threshold_db=THRESHOLD_DB)


def stage2_traffic():
    """DRAM bytes of one stage-2 k4 block from THIS round's ncu capture (tools/ncu_stage2_traffic.py writes the file from the
    --set full report); None when the capture is absent."""
    f = ROOT / 'profiles' / 'r02b_stage2_traffic.json'      # this round's latest `--set full` capture (tools/gpu_r02b_final.sh)
    if not f.exists():
        return None, None
    d = json.loads(f.read_text())
    return float(d['dram_bytes_per_forward']), d.get('source')


def measured_peaks():
    p = ROOT / 'MEASURED_PEAKS.json'
    if p.exists():
        d = json.loads(p.read_text())
        # the default timed region is short (K x ~0.3 ms at full clocks, ~200 W), nothing like the 1.3 GHz / 1 kW state of the sustained
        # cuBLAS figure: the BURST figure is the honest denominator (VERDICT r1); the sustained one is reported beside it
        return dict(tflops=float(d['bf16_tflops']), hbm=float(d['hbm_gbs']), burst=float(d['bf16_tflops']),
                    sustained=float(d.get('bf16_tflops_sustained') or d['bf16_tflops']),
                    source='measured (MEASURED_PEAKS.json, cuBLAS bf16 burst; sustained figure in peak_sustained)')
    return dict(tflops=1590.0, hbm=6650.0, burst=1590.0, sustained=1400.0, source='fallback (B200_PROFILING.md)')


class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop_evt = threading.Event()
        self.ready = threading.Event()

    def run(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.ready.set()
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            names = {
                getattr(pynvml, 'nvmlClocksEventReasonHwSlowdown', 0x8): 'hw_slowdown',
                getattr(pynvml, 'nvmlClocksEventReasonHwThermalSlowdown', 0x40): 'hw_thermal_slowdown',
                getattr(pynvml, 'nvmlClocksEventReasonSwThermalSlowdown', 0x20): 'sw_thermal_slowdown',
                getattr(pynvml, 'nvmlClocksEventReasonSwPowerCap', 0x4): 'sw_power_cap',
            }
            while not self._stop_evt.is_set():
                self.samples.append(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                try:
                    r = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    r = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
                time.sleep(0.005)
        except Exception as exc:        # clocks are best-effort; never fail the bench for them
            self.reasons.add(f'unavailable:{type(exc).__name__}')

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return dict(sm_mhz=med, sm_max_mhz=self.max_mhz, reasons=sorted(self.reasons))


def make_models(rank, world):
    """rank 0 writes the seeded synthetic model files; with N > 1 the arrays are NCCL-broadcast so that
    every rank uploads identical weights (the only collective of the whole job)."""
    from realtime_yukarin_b200 import synthetic
    d = Path(tempfile.mkdtemp(prefix=f'ryk_bench_r{rank}_'))
    if world == 1:
        return synthetic.write_synthetic_models(d, seed=0)
    from realtime_yukarin_b200.distributed import broadcast_params
    p1 = broadcast_params(synthetic.make_stage1_params(0) if rank == 0 else None, src=0, device='cuda')
    p2 = broadcast_params(synthetic.make_stage2_params(0) if rank == 0 else None, src=0, device='cuda')
    paths = synthetic.write_synthetic_models(d, seed=0, base1=8, base2=8)     # configs / statistics files
    np.savez(paths['stage1_model_path'], **p1)
    np.savez(paths['stage2_model_path'], **p2)
    return paths


class CpuPath:
    """The CPU implementation of the same path (oracle port: C WORLD/SPTK + torch-CPU convs), one stream."""

    def __init__(self, paths, stream=0, threads=None, n_chunks=64):
        import torch
        from oracle import nets as onets
        from oracle import pipeline as opipe
        from realtime_yukarin_b200 import synthetic
        if threads:
            torch.set_num_threads(threads)
        self.cores = torch.get_num_threads()
        p1, p2 = onets.load_npz(paths['stage1_model_path']), onets.load_npz(paths['stage2_model_path'])
        stats = (float(np.log(150.0)), 0.2, float(np.log(250.0)), 0.2)
        cfg = opipe.PathConfig(threshold_db=THRESHOLD_DB)
        self.orc = opipe.StreamOracle(cfg, p1, p2, stats, buffer_time=BUFFER_TIME, extra=EXTRA, backend='torch')
        self.n = round(BUFFER_TIME * FS)
        self.x = synthetic.synthetic_speech((n_chunks + 1) * BUFFER_TIME, stream=stream)
        self.k = 0

    def step(self):
        k = self.k % (len(self.x) // self.n)
        self.orc.push(self.x[k * self.n:(k + 1) * self.n])
        self.k += 1

    def rate(self, n_chunks):
        t0 = time.perf_counter()
        for _ in range(n_chunks):
            self.step()
        return n_chunks / (time.perf_counter() - t0)


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def run_reference_worker(args):
    """One CPU stream of the reference arm (child process of run_reference): prints {"dt": seconds for `steps` chunks, "cores": threads}."""
    from realtime_yukarin_b200 import synthetic
    d = Path(tempfile.mkdtemp(prefix=f'ryk_ref_w{args.stream}_'))
    paths = synthetic.write_synthetic_models(d, seed=0)
    cpu = CpuPath(paths, stream=args.stream, threads=args.threads, n_chunks=args.steps + args.warmup + 1)
    for _ in range(max(1, args.warmup)):
        cpu.step()
    print(json.dumps(dict(ready=True)), flush=True)
    sys.stdin.readline()                                  # all workers start their timed chunks together
    t1 = time.perf_counter()
    for _ in range(args.steps):
        cpu.step()
    print(json.dumps(dict(dt=time.perf_counter() - t1, cores=cpu.cores)), flush=True)


def run_reference(args):
    """The CPU implementation of the path on the host cores.  N = 1: one stream, all cores.  N > 1 (under torchrun): rank 0 alone
    does the work (the other ranks exit 0) -- it runs N independent streams, the job the N-GPU arm does, as N worker processes
    with cores / N threads each (torchrun's OMP_NUM_THREADS=1 is overridden), and reports their SUM: N * steps chunks over the
    slowest worker's time.  The ratio to the N-GPU arm is then whole job against whole job on the same box."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    import subprocess
    world = int(os.environ.get('WORLD_SIZE', str(args.gpus)))
    n_streams = max(1, world)
    cores = host_cores()
    threads = max(1, cores // n_streams)
    t0 = time.perf_counter()
    env = dict(os.environ)
    for k in ('OMP_NUM_THREADS', 'MKL_NUM_THREADS', 'RANK', 'LOCAL_RANK', 'WORLD_SIZE', 'MASTER_ADDR', 'MASTER_PORT', 'TORCHELASTIC_RUN_ID'):
        env.pop(k, None)
    env['OMP_NUM_THREADS'] = str(threads)
    procs = [subprocess.Popen([sys.executable, str(ROOT / 'bench.py'), '--impl', 'reference-worker', '--stream', str(i), '--threads', str(threads),
                               '--steps', str(args.steps), '--warmup', str(args.warmup)], stdin=subprocess.PIPE, stdout=subprocess.PIPE, env=env, text=True)
             for i in range(n_streams)]
    for pr in procs:                                       # warm-up done everywhere
        assert json.loads(pr.stdout.readline()).get('ready')
    for pr in procs:
        pr.stdin.write('go\n'); pr.stdin.flush()
    res = [json.loads(pr.stdout.readline()) for pr in procs]
    for pr in procs:
        pr.wait()
    dt = max(r['dt'] for r in res)
    used = sum(r['cores'] for r in res)
    value = n_streams * args.steps / dt
    line = dict(
        impl='reference', metric=METRIC, value=value, unit='chunks/s', rtf=value * BUFFER_TIME, n_gpus=args.gpus, steps=args.steps,
        warmup=args.warmup, ms_per_step=1000.0 * dt / args.steps, higher_is_better=True, scaling='weak', vs_baseline=None,
        dtype='f64 (WORLD/SPTK) + f32 (U-Nets)', data='synthetic',
        config=bench_config(WORKLOAD),
        reference_note='reference arm = CPU restatement of the path (C WORLD/SPTK + torch-CPU U-Nets) on the host cores; the reference itself cannot '
                       'run: its arithmetic lives in un-vendored pyworld/pysptk/chainer (SURVEY 8c).  One step = one 0.3 s chunk of every stream; '
                       f'{n_streams} independent stream(s) as {n_streams} process(es) x {threads} thread(s)',
        cpu_baseline=dict(value=value, unit='chunks/s', cores=used, kind='port',
                          sample=f'{args.steps} consecutive 0.3 s chunks of each of {n_streams} stream(s) after {max(1, args.warmup)} warm-up chunk(s); '
                                 f'{n_streams} process(es) x {threads} thread(s) on {cores} host cores'),
        e2e=dict(value=value, unit='chunks/s', h2d_bytes_per_step=0, d2h_bytes_per_step=0),
        wall_s=time.perf_counter() - t0)
    print(json.dumps(line))


def run_gpu(args):
    import torch
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    from realtime_yukarin_b200 import synthetic
    from realtime_yukarin_b200.engine import Engine, SessionConfig
    from realtime_yukarin_b200.models import AcousticConverter, F0Converter, SuperResolution
    from realtime_yukarin_b200.params import create_from_json, create_sr_from_json

    paths = make_models(rank, world)
    eng = Engine(device=local_rank)
    f0c = F0Converter(paths['input_statistics_path'], paths['target_statistics_path'])
    AcousticConverter(create_from_json(paths['stage1_config_path']), paths['stage1_model_path'], f0_converter=f0c, engine=eng)
    SuperResolution(create_sr_from_json(paths['stage2_config_path']), paths['stage2_model_path'], engine=eng)
    eng.set_precision('fp16')

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()
        eng.synchronize()

    def max_over_ranks(v):
        if world == 1:
            return v
        import torch.distributed as dist
        t = torch.tensor([v], dtype=torch.float64, device='cuda')
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def window(T):
        Tw = round((T + 2 * EXTRA[1]) * 200)
        return Tw, Tw + (128 - Tw % 128)

    def run_config(T, B, steps, warmup, with_e2e, sustain_s=0.0, f0_method='dio', dump_dir=None):
        """One workload (buffer_time T, B grouped streams per GPU) on every rank: device-resident leg, optional sustained repeat of
        the same K-step block, optional end-to-end leg with host buffers.  Returns a dict of rank-0 figures (times max over ranks)."""
        Tw, Tp = window(T)
        eng.set_f0_method(f0_method)          # sessions take the extractor that is selected when they are created

        def new_streams():
            """B sessions of this rank; B > 1: grouped so that stage 2 runs once per step at batch B (BASELINE config 5)."""
            def new_session():
                cfg = SessionConfig(fs=FS, frame_period_ms=5.0, f0_floor=71.0, f0_ceil=800.0, fft_length=1024, order=8, alpha=0.466,
                                    buffer_time=T, encode_extra_time=EXTRA[0], convert_extra_time=EXTRA[1], decode_extra_time=EXTRA[2],
                                    threshold_db=THRESHOLD_DB, vocoder_buffer_size=1024)
                return eng.session_create(cfg)
            sids = [new_session() for _ in range(B)]
            return sids, (eng.group_create(sids) if B > 1 else None)

        def free_streams(sids, gid):
            if gid is not None:
                eng.group_destroy(gid)
            for sid in sids:
                eng.session_destroy(sid)

        n = round(T * FS)
        total = warmup + steps
        xs = [synthetic.synthetic_speech((total + 1) * T, stream=rank * B + j) for j in range(B)]
        chunks = [[np.ascontiguousarray(x[k * n:(k + 1) * n]) for x in xs] for k in range(total)]     # [step][stream]

        # ---- leg 1: device-resident ("value") ----
        sids, gid = new_streams()
        d_in = torch.from_numpy(np.stack([np.stack(c) for c in chunks])).cuda()       # [step][stream][n]
        out_cap = (n // 1024 + 5) * 1024 + 8192
        RING = 8                                     # distinct output slots: consecutive chunks are in flight together
        d_out = torch.empty((RING, B, out_cap), dtype=torch.float64, device='cuda')
        d_n = torch.zeros((RING, B), dtype=torch.int32, device='cuda')

        def push_dev(k):
            r, ki = k % RING, k % total
            if gid is None:
                eng.session_push_device(sids[0], d_in[ki, 0].data_ptr(), n, d_out[r, 0].data_ptr(), out_cap, d_n[r, 0:].data_ptr())
            else:
                eng.group_push_device(gid, [d_in[ki, j].data_ptr() for j in range(B)], n, [d_out[r, j].data_ptr() for j in range(B)], out_cap,
                                      [d_n[r, j:].data_ptr() for j in range(B)])

        eng.profile(True)                            # warm up the same (event-instrumented) graphs the timed region replays
        for k in range(warmup):
            push_dev(k)
        barrier()
        eng.profile_read2()                          # discard the warm-up timings
        sampler = ClockSampler(local_rank)
        sampler.start()
        sampler.ready.wait(timeout=5)
        launches0 = eng.launch_count
        eng.profile(True)
        eng.timer_start()
        t_host0 = time.perf_counter()
        trace = []
        for k in range(warmup, total):
            push_dev(k)
            trace.append(time.perf_counter())
        if os.environ.get('RYK_BENCH_TRACE') == '1':
            print('host us per push:', [round((b - a) * 1e6) for a, b in zip([t_host0] + trace[:-1], trace)], file=sys.stderr)
        t_host = time.perf_counter() - t_host0          # host time to queue the K steps (launch overhead view)
        t_dev = eng.timer_stop() * 1e-3          # CUDA events on the stream the kernels are launched on
        barrier()
        s2_sum, s2_ms, s2_runs = eng.profile_read2()   # s2_ms = union of the per-forward intervals (consecutive forwards overlap on two streams)
        eng.profile(False)
        clocks = sampler.stop()
        if dump_dir is not None:
            # the waveform every stream's caller received from the last timed push, read before the sustained leg reuses the ring slots;
            # a stream whose share of DUMP_BYTES it would exceed is written as every k-th sample, the smallest k that fits
            r = (total - 1) % RING
            counts = d_n[r].cpu().numpy()
            cap = max(1, DUMP_BYTES // (8 * world * B))
            for j in range(B):
                wave = d_out[r, j, :int(counts[j])].cpu().numpy().astype(np.float64)
                np.save(dump_dir / f'wave_rank{rank}_stream{j}.npy', wave[::-(-len(wave) // cap)] if len(wave) > cap else wave)
        launches = eng.launch_count - launches0
        res = dict(T=T, B=B, Tw=Tw, Tp=Tp, n=n, t_dev=max_over_ranks(t_dev), t_host=t_host, s2_ms=s2_ms, s2_sum=s2_sum, s2_runs=s2_runs, launches=launches, clocks=clocks)

        # ---- sustained: the same K-step block repeated back to back for >= sustain_s seconds (thermal / power steady state) ----
        if sustain_s > 0:
            sampler = ClockSampler(local_rank)
            sampler.start()
            sampler.ready.wait(timeout=5)
            rates, s2_tot, s2_n = [], 0.0, 0
            t_wall = time.perf_counter()
            k = total
            while time.perf_counter() - t_wall < sustain_s:
                eng.profile(True)
                eng.timer_start()
                for _ in range(steps):
                    push_dev(k)
                    k += 1
                dt = eng.timer_stop() * 1e-3
                _sum, a, b_ = eng.profile_read2()
                s2_tot += a; s2_n += b_
                rates.append(B * steps / dt)
            eng.profile(False)
            barrier()
            res['sustained'] = dict(rates=rates, seconds=time.perf_counter() - t_wall, clocks=sampler.stop(), s2_ms=s2_tot, s2_runs=s2_n)
        if os.environ.get('RYK_STAGE_TIMES') == '1':       # diagnostics: device time of each stage of the last pipelined step
            st, en = eng.session_stage_times(sids[0])
            res['stage_times'] = dict(stages=['gate_slides', 'world_analysis', 'stage1', 'stage2', 'synthesis'],
                                      start_ms=np.round(st, 3).tolist(), end_ms=np.round(en, 3).tolist())
        free_streams(sids, gid)
        del d_in, d_out, d_n

        # ---- leg 2: end to end with host buffers ("e2e") ----
        if with_e2e:
            sids, gid = new_streams()
            host_out = [np.empty(out_cap, dtype=np.float64) for _ in range(B)]
            produced = 0
            DEPTH = 4                                    # steps in flight (submit k, collect k - DEPTH; the API allows 5): host buffers both ways

            def submit(k):
                return eng.session_submit(sids[0], chunks[k][0]) if gid is None else eng.group_submit(gid, chunks[k])

            def collect(t):
                if gid is None:
                    return len(eng.session_collect(sids[0], t, host_out[0]))
                return sum(len(o) for o in eng.group_collect(gid, t, host_out))

            for k in range(warmup):
                collect(submit(k))
            barrier()
            t0 = time.perf_counter()
            tickets = []
            for k in range(warmup, total):
                tickets.append(submit(k))
                if len(tickets) > DEPTH:
                    produced += collect(tickets.pop(0))
            while tickets:
                produced += collect(tickets.pop(0))
            t_e2e = time.perf_counter() - t0
            barrier()
            res['t_e2e'] = max_over_ranks(t_e2e)
            res['produced'] = produced
            free_streams(sids, gid)
        eng.set_f0_method('dio')
        return res

    T, B = args.buffer_time, args.streams_per_gpu
    default_workload = (B == 1 and abs(T - BUFFER_TIME) < 1e-9)
    dump_dir = None
    if args.dump_outputs:
        dump_dir = Path(args.dump_outputs)
        dump_dir.mkdir(parents=True, exist_ok=True)
    main = run_config(T, B, args.steps, args.warmup, with_e2e=True, sustain_s=(args.sustain if default_workload else 0.0), dump_dir=dump_dir)
    extras = []
    if default_workload and not args.no_extra:
        # BASELINE configs 3 and 5, short device-resident legs so that the driver's N = 1..8 runs record them too
        for (Tx, Bx, sx) in EXTRA_LEGS:
            extras.append(run_config(Tx, Bx, sx, 3, with_e2e=False))
        # the default workload with Harvest (+ StoneMask) as the f0 extractor inside the session's analysis graph (north_star: "DIO/Harvest f0")
        harvest_leg = run_config(T, 1, 12, 3, with_e2e=False, f0_method='harvest')

    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    peaks = measured_peaks()

    def tflops(r):
        return stage2_tc_flop(r['Tp']) * r['B'] * r['s2_runs'] / (r['s2_ms'] * 1e-3) / 1e12 if r['s2_ms'] > 0 else None

    Tw, Tp, n = main['Tw'], main['Tp'], main['n']
    value = world * B * args.steps / main['t_dev']
    e2e = world * B * args.steps / main['t_e2e']
    fl = stage2_tc_flop(Tp) * B
    ach = tflops(main)
    cpu_rate = cores = None
    if world == 1 and default_workload:                      # reported baseline: rank 0 at N = 1 only
        cpu = CpuPath(paths, n_chunks=8)
        cpu.step()
        cpu_rate, cores = cpu.rate(3), cpu.cores
    metric = METRIC if default_workload else f'chunks_per_s_{T:g}s_24kHz_encode_stage1_stage2_vocode'

    def workload_of(T_, B_, Tw_, Tp_):
        return (f'{B_} stream(s) per GPU' + (' grouped: one batched stage-2 forward per step' if B_ > 1 else '') +
                f', buffer_time={T_:g} s, extras (0,0.5,0), frame_period 5 ms, 24 kHz in/out, convert window {Tw_} -> {Tp_} frames, '
                f'stage-2 input ({B_},1,{Tp_},512), same models as the default workload; one step = one chunk of every stream')
    workload = WORKLOAD if default_workload else workload_of(T, B, Tw, Tp)
    traffic, traffic_src = stage2_traffic() if default_workload else (None, None)
    line = dict(
        metric=metric, value=value, unit='chunks/s', rtf=value * T, n_gpus=world, steps=args.steps, warmup=args.warmup,
        ms_per_step=1000.0 * main['t_dev'] / args.steps, higher_is_better=True, scaling='weak', vs_baseline=None,
        dtype=DTYPE, data='synthetic',
        config=bench_config(workload, B),
        e2e=dict(value=e2e, unit='chunks/s', rtf=e2e * T, h2d_bytes_per_step=B * n * 4,
                 d2h_bytes_per_step=int(main['produced'] / max(1, args.steps)) * 8 + B * (4 + 8)),
        gpu_launches=int(main['launches']), host_enqueue_ms_per_step=1000.0 * main['t_host'] / args.steps,
        clocks=main['clocks'],
        roofline=dict(bound='tensor', kernel=('stage-2 k4 layers 1..14: k_conv_tc (tcgen05, one tile per CTA) + k_splitk_reduce for c3-d3' if B == 1 else
                                              'stage-2 k4 layers 1..14: k_conv_halo (persistent tcgen05, c1-c3 / d3-d6) + k_conv_tc / k_splitk_reduce (c4-d2)'
                                              ' + the two 3x3 edge layers (group forward timed as a whole)'), achieved=ach, peak=peaks['tflops'],
                      unit='TFLOP/s', frac=(ach / peaks['tflops']) if ach else None, traffic=traffic, traffic_source=traffic_src,
                      peak_source=peaks['source'], peak_burst=peaks['burst'], peak_sustained=peaks['sustained'],
                      flop_per_step=fl, ms_per_step_in_kernel=(main['s2_ms'] / main['s2_runs']) if main['s2_runs'] else None,
                      ms_per_forward_wall=(main['s2_sum'] / main['s2_runs']) if main['s2_runs'] else None,
                      timed='CUDA events around the 14-layer graph of every forward on the stream it runs on, inside the pipelined timed region (co-running '
                            'stages included).  A session alternates its forwards between two streams, so consecutive forwards overlap: '
                            'ms_per_step_in_kernel = union of the intervals / forwards (time during which the block runs, per forward; `achieved` uses it), '
                            'ms_per_forward_wall = mean first-kernel-start to last-kernel-end of ONE forward'),
    )
    if 'sustained' in main:
        su = main['sustained']
        rates = sorted(su['rates'])
        s_ach = (stage2_tc_flop(Tp) * B * su['s2_runs'] / (su['s2_ms'] * 1e-3) / 1e12) if su['s2_ms'] > 0 else None
        line['sustained'] = dict(value=world * rates[len(rates) // 2], unit='chunks/s', seconds=su['seconds'], blocks=len(rates), steps_per_block=args.steps,
                                 min=world * rates[0], max=world * rates[-1], clocks=su['clocks'], stage2_tflops=s_ach,
                                 stage2_frac_of_sustained_peak=(s_ach / peaks['sustained']) if s_ach else None,
                                 note='median over back-to-back K-step blocks on rank 0 x N ranks (every rank runs the same loop)')
    if extras:
        ex = {}
        for r, (Tx, Bx, sx) in zip(extras, EXTRA_LEGS):
            v = world * Bx * sx / r['t_dev']
            a = tflops(r)
            ex[f'{Bx}x{Tx:g}s'] = dict(value=v, unit='chunks/s', rtf=v * Tx, steps=sx, ms_per_step=1000.0 * r['t_dev'] / sx, streams_per_gpu=Bx,
                                       workload=workload_of(Tx, Bx, r['Tw'], r['Tp']), stage2_tflops=a,
                                       stage2_frac=(a / peaks['tflops']) if a else None)
        vh = world * 12 / harvest_leg['t_dev']
        ex['1x0.3s_harvest_f0'] = dict(value=vh, unit='chunks/s', rtf=vh * T, steps=12, ms_per_step=1000.0 * harvest_leg['t_dev'] / 12, streams_per_gpu=1,
                                       workload=workload_of(T, 1, harvest_leg['Tw'], harvest_leg['Tp']) + ', f0 = Harvest + StoneMask')
        line['extra_configs'] = ex
    if 'stage_times' in main:
        line['stage_timeline'] = main['stage_times']
    if cpu_rate is not None:
        line['cpu_baseline'] = dict(value=cpu_rate, unit='chunks/s', cores=cores, kind='port',
                                    sample='3 chunks of 0.3 s after a warm-up chunk, C WORLD/SPTK restatement + torch-CPU U-Nets, same models/audio')
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=None)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference', 'reference-worker'])
    ap.add_argument('--stream', type=int, default=0, help='(reference-worker) stream index')
    ap.add_argument('--threads', type=int, default=None, help='(reference-worker) torch threads')
    ap.add_argument('--streams-per-gpu', type=int, default=1, help='B > 1: BASELINE config 5 style, B grouped streams per GPU')
    ap.add_argument('--buffer-time', type=float, default=BUFFER_TIME, help='seconds per chunk (default workload: 0.3)')
    ap.add_argument('--sustain', type=float, default=2.0, help='seconds of back-to-back K-step blocks for the `sustained` key (0 = skip)')
    ap.add_argument('--no-extra', action='store_true', help='skip the short BASELINE config 3 / 5 legs (`extra_configs`)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write the float64 waveform each stream produced in the last timed step as '
                         'DIR/wave_rank<r>_stream<j>.npy, at most 64 MB in all (a longer wave is written as every k-th sample); '
                         'inputs and weights are seeded: equal arguments give equal inputs')
    args = ap.parse_args()
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs writes what the timed GPU path computed; it applies to --impl b200 only')
    if args.steps is None:
        args.steps = 20 if args.impl == 'b200' else 6
    args.warmup = max(args.warmup, 3) if args.impl == 'b200' else args.warmup
    if args.impl == 'reference-worker':
        run_reference_worker(args)
    elif args.impl == 'reference':
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == '__main__':
    main()
