#!/usr/bin/env python3
"""bench.py -- stream-updates/s of the Precise streaming-inference hot path on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--streams-per-gpu S] [--impl b200|reference] [--dump-outputs DIR]

One "step" = one tick: every stream on the GPU receives one 1024-sample (2048-byte) chunk and is
fully classified: PCM -> MFCC frames -> 29-step GRU scan -> sigmoid -> threshold decode -> trigger
(+ for N > 1 the NCCL all-reduce of the detection count).  A (stream, chunk) pair is one
stream-update; ``value`` = stream-updates/s over all GPUs, weak scaling (S streams per GPU).

Workload (``config.workload``): the per-GPU shard of BASELINE.json configs[3] (1M default-parameter
streams over 8 GPUs; 131072 = 2^17 streams per GPU so that one tick's PCM, 268 MB, exceeds the
126 MB L2), default 'hey-mycroft' parameters (n_fft 512, 20 filters, 13 MFCCs, GRU 20).  configs[1]
(1k streams) is reported beside it under ``small_batch`` with an explicit L2 flush between steps.
Synthetic data: Gaussian sigma=3000 LSB int16 PCM, 1 % silent and 1 % full-scale-DC streams, seeded
random weights (no trained model ships with the reference).

The JSON line carries ``roofline`` (MFCC kernel vs measured HBM bandwidth; per-launch time from CUDA
events inside the timed region), ``roofline_gru`` (fp32-FMA bound scan kernel), ``e2e`` (same metric
through the host-buffer C-ABI call, pinned host PCM in / confidences out inside the timed region),
``cpu_baseline`` (the numpy oracle port on the host cores) and ``clocks``.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

# one BLAS / OpenMP thread per process (BASELINE.md section 3: "OMP_NUM_THREADS=1 per worker"); must be set before numpy loads its BLAS
for _v in ('OMP_NUM_THREADS', 'OPENBLAS_NUM_THREADS', 'MKL_NUM_THREADS', 'NUMEXPR_NUM_THREADS'):
    os.environ[_v] = '1'

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True    # the benchmark leaves the tree as it found it (which may be read-only): no __pycache__ from its imports

CHUNK = 1024
PRIME = 24                # ticks that fill a 29-frame window: (24 * 1024 - 1600) // 800 + 1 = 29 frames
ALG_BYTES_PER_UPDATE = 2048 + 1.28 * 13 * 4           # SURVEY 8d: 2114.56 B (F=13)
ALG_FLOP_PER_UPDATE_GRU = 2 * (29 * (13 + 20) * 60 + 20)   # 114 880
FP32_PEAK_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12     # 74.4 (148 SMs x 128 lanes x 2 x max clock)
K2_BYTES_PER_UPDATE = 29 * 240 + 4 + 8 + 1 + 8 + 1.28 * (52 + 240)   # 29 cached projection rows + raw, conf, fired, trigger state + the tick's new frames (MFCC row in, projection out)
K2_MMA_FLOP_PER_UPDATE = 29 * 27 * (4096 + 2048) // 16   # per 16-stream tile and step 27 m16n8k16 + 27 m16n8k8 fp16 MMAs (fp16x3 split included)
K1_NAMES = {0: 'mfcc_tc3_plan_kernel + mfcc_tc3_kernel (K1: int16 split exactly into fp16 pieces, both DFT stages on tcgen05 / TMEM) -- default from 49152 streams per tick',
            2: 'mfcc_fast_stream_kernel<LEAN> (K1, FFT on the CUDA cores)', 3: 'mfcc_fast_stream_kernel (K1, FFT, 64-bit set-up)',
            4: 'mfcc_tc2_stream_kernel (K1, DFT stage 2 on tcgen05)', 5: 'mfcc_tc3_plan_kernel + mfcc_tc3_kernel (K1, both DFT stages on tcgen05)'}


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.isfile(p):
        try:
            return float(json.load(open(p))['hbm_gbs']), 'measured'
        except Exception:
            pass
    return 6650.0, 'fallback'


def synth_pcm(n_streams, n_samples, seed, stream_offset=0):
    """Gaussian sigma=3000 int16; 1 % silent, 1 % DC streams (the reference's own test signals)."""
    rs = np.random.RandomState(seed)
    x = rs.standard_normal((n_streams, n_samples)).astype(np.float32)
    x *= 3000.0
    pcm = np.clip(x, -32768, 32767).astype(np.int16)
    ids = np.arange(n_streams) + stream_offset
    pcm[ids % 100 == 17] = 0
    pcm[ids % 100 == 53] = 32767
    return pcm


# ------------------------------------------------------------------------------------ CPU arm
def workload_config(S, world, l2=None):
    """The ``config`` object of both arms (same keys and workload text, so that the two lines describe the same job)."""
    return {'workload': 'per-GPU shard of configs[3]: %d streams/GPU x %d GPU, default hey-mycroft parameters '
                        '(n_fft 512, hop 800, window 1600, n_filt 20, n_mfcc 13, GRU 20, 29-frame window), 1024-sample chunks' % (S, world),
            'streams_per_gpu': S, 'chunk_samples': CHUNK,
            'priming': '%d untimed ticks before the warm-up fill every 29-frame window: each timed update scans 29 real frames' % PRIME,
            'l2': l2 or 'inputs larger than L2',
            'parallelism': 'streams block-sharded over GPUs, NCCL all-reduce of the detection count per tick (on a side stream, under the next tick)' if world > 1 else 'single GPU'}


def _limit_threads():
    """One BLAS/OpenMP thread in this process; fails loudly if that cannot be enforced."""
    from threadpoolctl import threadpool_limits, threadpool_info
    threadpool_limits(1)
    bad = [i for i in threadpool_info() if i.get('num_threads', 1) != 1]
    if bad:
        raise RuntimeError('could not pin BLAS/OpenMP to one thread: %r' % bad)


def _cpu_worker_loop(conn, seed, warm):
    """One Listener per process, as the reference runs it (precise/network_runner.py:101-153 + runner.py:127-142): the numpy oracle
    port of Listener.update + TriggerDetector.update on one stream.  Warm-up once (window filled, caches hot), then timed batches."""
    _limit_threads()
    from oracle.gru import GruWeights
    from oracle.listener import OracleListener
    from oracle.trigger import OracleTrigger
    w = GruWeights.random(13, 20, seed=0, scale=0.1)
    ring = 256
    pcm = synth_pcm(1, ring * CHUNK, seed)[0]
    chunks = [pcm[k * CHUNK:(k + 1) * CHUNK].astype(np.float32) / 32768.0 for k in range(ring)]
    lis, det = OracleListener(w), OracleTrigger(2 * CHUNK)
    k = 0
    for _ in range(warm):
        det.update(lis.update(chunks[k % ring])); k += 1
    conn.send('ready')
    while True:
        cmd = conn.recv()
        if cmd is None:
            return
        ticks = int(cmd)
        fired = 0
        t0 = time.perf_counter()
        for _ in range(ticks):
            fired += det.update(lis.update(chunks[k % ring])); k += 1
        conn.send((ticks, time.perf_counter() - t0, fired))


class CpuPool:
    """Persistent worker processes (one stream each, one core each, 50 warm-up ticks at start)."""
    WARM = 50

    def __init__(self, procs=None):
        import multiprocessing as mp
        self.procs = procs or usable_cores()
        ctx = mp.get_context('fork')
        self.w = []
        for i in range(self.procs):
            a, b = ctx.Pipe()
            p = ctx.Process(target=_cpu_worker_loop, args=(b, 1000 + i, self.WARM), daemon=True)
            p.start()
            self.w.append((p, a))
        for _, a in self.w:
            assert a.recv() == 'ready'

    def step(self, ticks):
        """Every worker runs `ticks` timed ticks concurrently -> (stream-updates, wall seconds = slowest worker)."""
        for _, a in self.w:
            a.send(ticks)
        res = [a.recv() for _, a in self.w]
        return sum(r[0] for r in res), max(r[1] for r in res)

    def close(self):
        for p, a in self.w:
            try:
                a.send(None)
            except Exception:
                pass
        for p, _ in self.w:
            p.join(timeout=5)


def cpu_port_rate(ticks=1000, steps=3, pool=None):
    """The oracle port on all usable host cores: `steps` batches of `ticks` (>= 1000, BASELINE.md section 3) timed ticks per worker
    after 50 warm-up ticks per worker -> (stream-updates/s, workers, description, wall seconds per step)."""
    own = pool is None
    pool = pool or CpuPool()
    try:
        upd = wall = 0.0
        for _ in range(steps):
            u, t = pool.step(ticks)
            upd += u; wall += t
    finally:
        if own:
            pool.close()
    return upd / wall, pool.procs, ('%d worker processes x 1 stream x %d x %d timed ticks of 1024 samples (after %d warm-up ticks per worker, persistent '
                                    'workers), numpy oracle port of Listener.update + TriggerDetector.update, OMP/BLAS threads = 1 per worker'
                                    % (pool.procs, steps, ticks, CpuPool.WARM)), wall / steps


def cpu_c_port_rate(streams_per_thread=48, ticks=80):
    """The plain-C restatement (oracle/c/precise_oracle.c), streams sharded over one thread per usable core."""
    from oracle.cport import COracle
    from oracle.gru import GruWeights
    from oracle.params import OracleParams
    threads = usable_cores()
    co = COracle(GruWeights.random(13, 20, seed=0, scale=0.1), OracleParams(), chunk_samples=CHUNK)
    S = streams_per_thread * threads
    pcm = synth_pcm(S, ticks * CHUNK, 2468)
    co.run_streams(pcm[:threads, :4 * CHUNK], threads=threads)            # warm-up
    t0 = time.perf_counter()
    co.run_streams(pcm, threads=threads)
    dt = time.perf_counter() - t0
    return S * ticks / dt, threads, '%d threads x %d streams x %d ticks of 1024 samples, scalar C restatement (gcc -O2), float64 MFCC / float32 GRU' % (
        threads, streams_per_thread, ticks)


def _cpu_batched_worker(args):
    """The batched offline pattern of the reference (precise/scripts/simulate.py:92-104): vectorize a whole recording, cut one
    29-frame window per chunk_size // hop_samples frames, Runner.predict on [N, 29, 13]."""
    seed, seconds = args
    _limit_threads()
    from oracle import mfcc as om
    from oracle.gru import GruWeights, predict
    from oracle.params import OracleParams
    pr = OracleParams()
    w = GruWeights.random(13, 20, seed=0, scale=0.1)
    audio = synth_pcm(1, int(seconds * 16000), seed)[0].astype(np.float32) / 32768.0
    hops = max(1, CHUNK // pr.hop_samples)
    t0 = time.perf_counter()
    mf = om.vectorize_raw(audio, pr)
    inputs = np.array([mf[i - pr.n_features:i] for i in range(pr.n_features, len(mf), hops)])
    p = predict(w, inputs)
    return len(p), time.perf_counter() - t0, seconds


def cpu_batched_rate(seconds=120.0):
    import multiprocessing as mp
    procs = usable_cores()
    ctx = mp.get_context('fork')
    with ctx.Pool(procs) as pool:
        pool.map(_cpu_batched_worker, [(i, 5.0) for i in range(procs)])              # warm-up
        res = pool.map(_cpu_batched_worker, [(2000 + i, seconds) for i in range(procs)])
    wall = max(r[1] for r in res)
    return {'value': sum(r[0] for r in res) / wall, 'unit': 'window-predictions/s', 'realtime_streams': procs * seconds / wall, 'cores': procs,
            'kind': 'port', 'sample': '%d workers x %.0f s of audio: vectorize_raw on the whole recording, one 29 x 13 window per frame, '
                                      'batched GRU predict (simulate.py:92-104 pattern), numpy oracle port' % (procs, seconds)}


def usable_cores():
    """Host cores this process may actually use: affinity mask capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
    try:
        q, per = open('/sys/fs/cgroup/cpu.max').read().split()
        if q != 'max':
            n = max(1, min(n, int(float(q) / float(per) + 0.5)))
    except Exception:
        try:
            q = int(open('/sys/fs/cgroup/cpu/cpu.cfs_quota_us').read())
            per = int(open('/sys/fs/cgroup/cpu/cpu.cfs_period_us').read())
            if q > 0:
                n = max(1, min(n, int(q / per + 0.5)))
        except Exception:
            pass
    return n


def cpu_latency(calls=1000, warm=50):
    """p50/p99 of one oracle Listener.update + TriggerDetector.update (batch 1, one core), microseconds."""
    _limit_threads()
    from oracle.gru import GruWeights
    from oracle.listener import OracleListener
    from oracle.trigger import OracleTrigger
    w = GruWeights.random(13, 20, seed=0, scale=0.1)
    pcm = synth_pcm(1, (calls + warm) * CHUNK, 4321)
    lis, det = OracleListener(w), OracleTrigger(2 * CHUNK)
    ts = []
    for k in range(calls + warm):
        c = pcm[0, k * CHUNK:(k + 1) * CHUNK].astype(np.float32) / 32768.0
        t0 = time.perf_counter()
        det.update(lis.update(c))
        ts.append(time.perf_counter() - t0)
    ts = np.array(ts[warm:]) * 1e6
    return float(np.percentile(ts, 50)), float(np.percentile(ts, 99))


def host_info():
    model = None
    try:
        for ln in open('/proc/cpuinfo'):
            if ln.startswith('model name'):
                model = ln.split(':', 1)[1].strip()
                break
    except Exception:
        pass
    return {'os_cpu_count': os.cpu_count(), 'usable_cores': usable_cores(), 'cpu_model': model,
            'threads_per_worker': {v: os.environ.get(v) for v in ('OMP_NUM_THREADS', 'OPENBLAS_NUM_THREADS', 'MKL_NUM_THREADS')}}


def run_reference(args, rank):
    """--impl reference: the reference's CPU path (numpy oracle port; the TF/Keras/sonopy stack is not installable on this image)
    on all usable host cores.  A step = 1000 timed ticks on every worker (one stream per worker process, persistent workers,
    50 warm-up ticks each: BASELINE.md section 3); value = stream-updates over all timed steps / their wall time."""
    if rank != 0:
        return
    TICKS = 1000
    pool = CpuPool()
    try:
        for _ in range(args.warmup):
            pool.step(TICKS)
        upd = wall = 0.0
        for _ in range(args.steps):
            u, t = pool.step(TICKS)
            upd += u; wall += t
    finally:
        pool.close()
    v = upd / wall
    sample = ('%d worker processes x 1 stream x %d timed ticks per step (after %d warm-up ticks per worker and %d warm-up steps), numpy oracle '
              'port, OMP/BLAS threads = 1 per worker' % (pool.procs, TICKS, CpuPool.WARM, args.warmup))
    try:                                           # extra evidence: the compiled scalar C restatement on the same cores
        cc = cpu_c_port_rate()
        cpu_c = {'value': cc[0], 'unit': 'stream-updates/s', 'cores': cc[1], 'kind': 'port', 'sample': cc[2]}
    except Exception as e:
        cpu_c = None
        print('note: C port baseline skipped: %r' % (e,), file=sys.stderr)
    try:
        batched = cpu_batched_rate(60.0)
    except Exception as e:
        batched = None
        print('note: batched CPU baseline skipped: %r' % (e,), file=sys.stderr)
    S = args.streams_per_gpu                       # the same `config` object as the b200 arm prints for these arguments
    cfg = workload_config(S, args.gpus, ('inputs larger than L2: %d MB of PCM per tick, %d distinct ticks resident' % (S * CHUNK * 2 >> 20, args.ticks_resident))
                          if S * CHUNK * 2 >= (160 << 20) else 'explicit 256 MB flush write between steps (its time measured separately and subtracted)')
    line = {
        'impl': 'reference', 'metric': 'stream-updates/s (16 kHz int16 PCM, 1024-sample chunk -> decoded confidence + trigger)',
        'value': v, 'unit': 'stream-updates/s', 'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': 1e3 * wall / max(1, args.steps),
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64 MFCC / f32 GRU', 'data': 'synthetic',
        'config': cfg,
        'cpu_baseline': {'value': v, 'unit': 'stream-updates/s', 'cores': pool.procs, 'kind': 'port', 'sample': sample,
                         'per_core': v / pool.procs},
        'e2e': {'value': v, 'unit': 'stream-updates/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'realtime_streams': v / 15.625,
        'sample': 'the CPU arm times a bounded sample of the per-stream work of `config`: ' + sample,
        'cpu_baseline_c': cpu_c,
        'cpu_baseline_batched': batched,
        'host': host_info(),
        'note': 'value = numpy oracle port (the reference itself is Python + numpy + Keras/TF per Listener); cpu_baseline_c = the same '
                'path as compiled scalar C, a stronger CPU baseline than the reference could reach; cpu_baseline_batched = the offline '
                'simulate.py pattern (whole-recording MFCC + batched predict)',
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = 'index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,' \
        'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile('w+', suffix='.csv', delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(['nvidia-smi', '-i', str(gpu_index), '--query-gpu=' + self.Q, '--format=csv,noheader,nounits', '-lms', '20'],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(', ') for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        for r in rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except ValueError:
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), r[5:9]):
                if v.strip().lower() == 'active':
                    reasons.add(name)
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))
        return out


# ------------------------------------------------------------------------------------ GPU arm
DUMP_MAX_STREAMS = 1 << 21      # 24 B of .npy data per stream: a dump stays under 48 MB at any --streams-per-gpu


def last_tick_outputs(out, count):
    """Host copies of what one StreamBatch.update tick returns to its caller (raw network output, decoded confidence and trigger
    flag per stream) and of the detection count it accumulates.  Above DUMP_MAX_STREAMS streams a fixed, seeded sample of the
    streams is kept; ``stream`` holds the stream index of every row."""
    n = out['conf'].shape[0]
    idx = np.arange(n) if n <= DUMP_MAX_STREAMS else np.sort(np.random.RandomState(0).choice(n, DUMP_MAX_STREAMS, replace=False))
    return {'raw': out['raw'].cpu().numpy()[idx].astype(np.float32), 'conf': out['conf'].cpu().numpy()[idx].astype(np.float64),
            'fired': out['fired'].cpu().numpy()[idx].astype(np.float32), 'stream': idx.astype(np.float64),
            'detections': count.cpu().numpy().astype(np.float64)}


def run_b200(args):
    import torch
    import torch.distributed as dist
    from mycroft_precise_b200 import GruModel, StreamBatch
    from mycroft_precise_b200.core import pinned_empty, pinned_free
    from mycroft_precise_b200.dist import init_from_env, DetectionCounter, bind_to_gpu_numa_node

    cpu = None
    cpu_lat = None
    cpu_c = None
    cpu_batched = None
    if int(os.environ.get('WORLD_SIZE', '1')) == 1 and not args.no_cpu_baseline:
        cpu = cpu_port_rate()                  # before CUDA is initialised in this process (fork safety)
        cpu_lat = cpu_latency() if args.latency else None
        try:
            cpu_batched = cpu_batched_rate(60.0)
        except Exception as e:
            print('note: batched CPU baseline skipped: %r' % (e,), file=sys.stderr)
        try:
            cpu_c = cpu_c_port_rate()
        except Exception as e:                     # the C port is optional evidence; never fail the bench on it
            cpu_c = None
            print('note: C port baseline skipped: %r' % (e,), file=sys.stderr)
    rank, local, world = init_from_env()
    if world != args.gpus and rank == 0:
        print('note: WORLD_SIZE=%d, --gpus=%d' % (world, args.gpus), file=sys.stderr)
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    # CPU legs are done: from here on this process only feeds its GPU.  Pin it (and the pinned buffers it is about to allocate)
    # to the GPU's NUMA node, so that N ranks do not push their host traffic across the socket interconnect.
    numa_cpus = None if args.no_numa_bind else bind_to_gpu_numa_node(local)
    S = args.streams_per_gpu
    K, W = args.steps, args.warmup
    model = GruModel.random(13, 20, seed=0, scale=0.1)
    model.dense_b = 3.0          # confidence above the trigger threshold: the detection path and the count all-reduce carry real data
    sb = StreamBatch(model, S, chunk_samples=CHUNK, device=local)
    core = sb.core
    if args.gru_mode:
        core.gru_mode(args.gru_mode)
    if args.k1_mode:
        core.k1_mode(args.k1_mode)

    # ---- synthetic PCM: NT distinct ticks resident in HBM (each tick 2 KB x S > L2 at the default S)
    NT = args.ticks_resident
    host_ticks = [synth_pcm(S, CHUNK, seed=1234 + 17 * t, stream_offset=rank * S) for t in range(NT)]
    dev_ticks = [torch.from_numpy(h).to(dev) for h in host_ticks]
    counter = DetectionCounter(sb.count)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev) if S * CHUNK * 2 < (160 << 20) else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step(t):
        if flush is not None:
            flush.add_(1)                      # rewrite 256 MB: evicts L2 between iterations
        out = sb.update(dev_ticks[t % NT])
        if world > 1:
            counter.all_reduce_overlapped()    # snapshot on this stream, NCCL on a side stream under the next tick's K1
        return out

    # ---- value: inputs resident in HBM
    # Priming (untimed, before the warm-up): PRIME ticks fill every stream's 29-frame window, so that each timed update
    # scans 29 real frames (a stream younger than 29 frames reads fewer ring rows -- that would be skipped work).
    for t in range(PRIME):
        sb.update(dev_ticks[t % NT])
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None     # samples from here to the end of the e2e loop
    for t in range(W):
        step(t)
    barrier()
    core.profile(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    flush_ms = 0.0
    if flush is not None:                       # cost of the flush alone, subtracted below
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        for _ in range(K):
            flush.add_(1)
        f1.record(); torch.cuda.synchronize()
        flush_ms = f0.elapsed_time(f1)
        barrier()
    e0.record()
    for t in range(K):
        out = step(W + t)
    counter.wait()                              # the last tick's all-reduce is inside the timed region
    e1.record()
    barrier()
    # the last timed tick's results, copied before the e2e loop below advances the same streams
    dump = last_tick_outputs(out, counter.total if world > 1 else sb.count) if args.dump_outputs and rank == 0 else None
    ms = e0.elapsed_time(e1) - flush_ms
    kms, klaunch = core.profile_read()
    core.profile(False)
    tmax = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    ms_all = float(tmax.item())
    value = S * world * K / (ms_all * 1e-3)
    torch.cuda.synchronize()
    total_fired = int(counter.total.item()) if world > 1 else int(sb.count.item())

    # ---- e2e: host buffers through pb_update_host (H2D of the PCM and D2H of the results inside)
    pins = []
    e2e = None
    try:
        hp = []
        for t in range(min(NT, 2)):
            a, p = pinned_empty((S, CHUNK), np.int16); a[:] = host_ticks[t]; hp.append(a); pins.append(p)
        conf, p = pinned_empty((S,), np.float64); pins.append(p)
        fired, p = pinned_empty((S,), np.uint8); pins.append(p)
        for t in range(W):
            sb.update_host(hp[t % len(hp)], conf, None, fired)
        barrier()
        t0 = time.perf_counter()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        cnt = 0
        for t in range(K):
            cnt += sb.update_host(hp[t % len(hp)], conf, None, fired)
            if world > 1:
                counter.all_reduce_overlapped()
        counter.wait()
        g1.record()
        barrier()
        wall_ms = (time.perf_counter() - t0) * 1e3
        e_ms = g0.elapsed_time(g1)            # events bracket the blocking host calls: ~ wall time
        if e_ms <= 0:
            e_ms = wall_ms
        te = torch.tensor([e_ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e2e = {'value': S * world * K / (float(te.item()) * 1e-3), 'unit': 'stream-updates/s',
               'h2d_bytes_per_step': int(S * CHUNK * 2), 'd2h_bytes_per_step': int(S * (8 + 1) + 8),
               'api': 'pb_update_host (StreamBatch.update_host), pinned host buffers', 'ms_per_step': float(te.item()) / K}
    finally:
        for p in pins:
            pinned_free(p)
    clocks = sampler.stop() if sampler else None

    # ---- configs[1]: 1k streams, explicit L2 flush between steps
    small = None
    if rank == 0 and args.small_batch:
        S2 = 1000
        sb2 = StreamBatch(model, S2, chunk_samples=CHUNK, device=local)
        tk = [torch.from_numpy(synth_pcm(S2, CHUNK, seed=99 + t)).to(dev) for t in range(4)]
        fl = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
        evs = []
        for t in range(PRIME):
            sb2.update(tk[t % 4])
        for t in range(W + K):
            fl.add_(1)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); sb2.update(tk[t % 4]); b.record()
            if t >= W:
                evs.append((a, b))
        torch.cuda.synchronize()
        per = float(np.mean([a.elapsed_time(b) for a, b in evs]))
        small = {'workload': 'configs[1]: 1000 streams, GRU 20, 1 GPU', 'ms_per_step': per, 'value': S2 / (per * 1e-3),
                 'unit': 'stream-updates/s', 'l2': 'flushed (256 MB write) before every step'}
        sb2.core.close()

    # ---- configs[2]: 100k streams, GRU 128, n_mfcc = n_filt = 40 (tiled GRU kernel)
    big = None
    if rank == 0 and args.config3:
        from mycroft_precise_b200 import ListenerParams
        pr3 = ListenerParams(n_filt=40, n_mfcc=40)
        S3 = 100000
        m3 = GruModel.random(40, 128, seed=1, scale=0.1 / np.sqrt(128 / 20.0))
        sb3 = StreamBatch(m3, S3, params=pr3, chunk_samples=CHUNK, device=local)
        tk = [torch.from_numpy(synth_pcm(S3, CHUNK, seed=500 + t)).to(dev) for t in range(4)]
        for t in range(PRIME + 2):
            sb3.update(tk[t % 4])
        torch.cuda.synchronize()
        sb3.core.profile(True)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        n3 = 6
        for t in range(n3):
            sb3.update(tk[(t + 2) % 4])
        b.record(); torch.cuda.synchronize()
        kms3, kl3 = sb3.core.profile_read()
        per = a.elapsed_time(b) / n3
        flop3 = 2 * (29 * (40 + 128) * 384 + 128)
        big = {'workload': 'configs[2]: 100000 streams, GRU 128, n_filt = n_mfcc = 40, 1 GPU', 'ms_per_step': per,
               'value': S3 / (per * 1e-3), 'unit': 'stream-updates/s', 'k1_ms': kms3[0] / max(1, kl3[0]), 'k2_ms': kms3[1] / max(1, kl3[1]),
               'k2_fp32_frac': S3 * flop3 / (kms3[1] / max(1, kl3[1]) * 1e-3) / 1e12 / FP32_PEAK_TFLOPS,
               'l2': 'inputs larger than L2 (195 MB of PCM per tick)'}
        sb3.core.close()
        del tk

    # ---- configs[4]: latency mode, batch = 1 PER GPU: every rank runs one Engine.get_prediction-sized call at a time, concurrently
    lat = None
    if args.latency:
        sb1 = StreamBatch(model, 1, chunk_samples=CHUNK, device=local)
        one, p1 = pinned_empty((1, CHUNK), np.int16)
        c1, p2 = pinned_empty((1,), np.float64)
        src = synth_pcm(1, CHUNK * 64, 777 + rank)
        ts = []
        if world > 1:
            dist.barrier()
        for k in range(2200):                               # the first 200 calls (window filled after 24) are dropped below
            one[0] = src[0, (k % 64) * CHUNK:(k % 64 + 1) * CHUNK]
            t0 = time.perf_counter()
            sb1.update_host(one, c1)                        # H2D 2 KB -> K1 -> K2/K3 -> D2H 8 B, host-synchronous
            ts.append(time.perf_counter() - t0)
        ts = np.array(ts[200:]) * 1e6
        mine = torch.tensor([float(np.percentile(ts, 50)), float(np.percentile(ts, 99))], dtype=torch.float64, device=dev)
        allr = [torch.zeros_like(mine) for _ in range(world)]
        if world > 1:
            dist.all_gather(allr, mine)
        else:
            allr = [mine]
        per_rank = [[float(v[0]), float(v[1])] for v in allr]
        lat = {'workload': 'configs[4]: batch 1 per GPU on %d GPU(s), window->decision through pb_update_host (pinned 2 KB in, 8 B out), all ranks concurrently' % world,
               'p50_us': max(v[0] for v in per_rank), 'p99_us': max(v[1] for v in per_rank), 'per_rank_p50_p99_us': per_rank, 'calls': int(len(ts)),
               'aggregate': 'p50_us / p99_us = the slowest rank'}
        if cpu_lat:
            lat.update(cpu_p50_us=cpu_lat[0], cpu_p99_us=cpu_lat[1], cpu='oracle port, 1 core')
        pinned_free(p1); pinned_free(p2)
        sb1.core.close()

    if world > 1:
        dist.barrier()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    hbm_peak, which = peaks()
    k1_name = K1_NAMES.get(args.k1_mode, 'k1 mode %d' % args.k1_mode) if (args.k1_mode or S >= 49152) else K1_NAMES[2]
    k1_ms = kms[0] / max(1, klaunch[0])
    k2_ms = kms[1] / max(1, klaunch[1])
    k1_gbs = S * ALG_BYTES_PER_UPDATE / (k1_ms * 1e-3) / 1e9 if k1_ms > 0 else None
    proj_ms = (kms[3] / klaunch[3]) if klaunch[3] > 1 else 0.0          # slot 3 = the separate projection kernels (one launch = the initial rebuild of the cache)
    bf16_peak = None
    try:
        bf16_peak = float(json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))['bf16_tflops_sustained'])
    except Exception:
        pass
    traffic = None
    tp = os.path.join(ROOT, 'profiles', 'k1_traffic.json')
    if os.path.isfile(tp):
        try:
            traffic = json.load(open(tp)).get('bytes_per_launch')
        except Exception:
            traffic = None
    line = {
        'metric': 'stream-updates/s (16 kHz int16 PCM, 1024-sample chunk -> decoded confidence + trigger)',
        'value': value, 'unit': 'stream-updates/s', 'n_gpus': world, 'steps': K, 'warmup': W,
        'ms_per_step': ms_all / K, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32', 'data': 'synthetic',
        'config': workload_config(S, world, ('inputs larger than L2: %d MB of PCM per tick, %d distinct ticks resident' % (S * CHUNK * 2 >> 20, NT))
                                  if flush is None else 'explicit 256 MB flush write between steps (its time measured separately and subtracted)'),
        'realtime_streams': value / 15.625,
        'detections': total_fired,
        'roofline': {'kernel': k1_name, 'bound': 'hbm', 'achieved': k1_gbs, 'peak': hbm_peak, 'unit': 'GB/s',
                     'frac': (k1_gbs / hbm_peak) if k1_gbs else None, 'of': which, 'traffic': traffic,
                     'traffic_source': 'profiles/k1_traffic.json (one ncu --set full capture of this kernel, not a live counter)' if traffic else None,
                     'algorithmic_bytes_per_launch': S * ALG_BYTES_PER_UPDATE, 'ms_per_launch': k1_ms, 'launches': klaunch[0],
                     'note': 'ms_per_launch = one tick of K1 (for the tcgen05 path: plan kernel + main kernel, both inside the CUDA-event bracket)'},
        # K2 (scan over cached projections) against both of its ceilings: HBM for the bytes it must move (29 cached projection rows of
        # 240 B per update, the results, and the new frames' MFCC rows in / projections out) and the tensor pipe for the MMA FLOPs it
        # executes (fp16 x 3 split: 27 m16n8k16 + 27 m16n8k8 per 16 streams and step = 300 672 FLOP per update) against the measured
        # sustained fp16/bf16 tensor rate
        'roofline_k2': {'kernel': 'gru_mma16_kernel<20,13> (K2+K3: fp16x3 mma.sync scan over bulk-copy-staged cached projections, projects the tick\'s new frames itself)',
                        'ms_per_launch': k2_ms, 'launches': klaunch[1], 'input_projection_ms_per_launch': proj_ms or None,
                        'hbm': {'algorithmic_bytes_per_update': K2_BYTES_PER_UPDATE, 'achieved': S * K2_BYTES_PER_UPDATE / (k2_ms * 1e-3) / 1e9 if k2_ms > 0 else None,
                                'peak': hbm_peak, 'unit': 'GB/s', 'frac': S * K2_BYTES_PER_UPDATE / (k2_ms * 1e-3) / 1e9 / hbm_peak if k2_ms > 0 else None},
                        'tensor': {'executed_flop_per_update': K2_MMA_FLOP_PER_UPDATE, 'achieved': S * K2_MMA_FLOP_PER_UPDATE / (k2_ms * 1e-3) / 1e12 if k2_ms > 0 else None,
                                   'peak': bf16_peak, 'unit': 'TFLOP/s (fp16 MMA, executed incl. the 3x split)',
                                   'frac': (S * K2_MMA_FLOP_PER_UPDATE / (k2_ms * 1e-3) / 1e12 / bf16_peak) if (bf16_peak and k2_ms > 0) else None},
                        'algorithmic_flop_per_update': ALG_FLOP_PER_UPDATE_GRU},
        'e2e': e2e,
        'gpu_launches': int(sum(klaunch)) + (int(klaunch[0]) if (args.k1_mode in (0, 5) and S >= 49152) else 0),     # K1 on the tcgen05 path = plan kernel + main kernel
        'cpu_baseline': ({'value': cpu[0], 'unit': 'stream-updates/s', 'cores': cpu[1], 'kind': 'port', 'sample': cpu[2]} if cpu else None),
        'cpu_baseline_c': ({'value': cpu_c[0], 'unit': 'stream-updates/s', 'cores': cpu_c[1], 'kind': 'port', 'sample': cpu_c[2]} if cpu_c else None),
        'cpu_baseline_batched': cpu_batched,
        'host': dict(host_info(), numa_bound_cpus=(('%d CPUs of the GPU\'s NUMA node, %d..%d' % (len(numa_cpus), numa_cpus[0], numa_cpus[-1])) if numa_cpus else None)),
        'clocks': clocks,
        'small_batch': small,
        'latency': lat,
        'config3': big,
    }
    if big:
        big.pop('k2_fp32_frac', None)
    for name, a in (dump or {}).items():
        np.save(os.path.join(args.dump_outputs, name + '.npy'), a)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=50)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--streams-per-gpu', type=int, default=131072)
    ap.add_argument('--ticks-resident', type=int, default=8)
    ap.add_argument('--no-small-batch', dest='small_batch', action='store_false')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-latency', dest='latency', action='store_false')
    ap.add_argument('--no-config3', dest='config3', action='store_false')
    ap.add_argument('--no-numa-bind', action='store_true', help='do not pin the process to the CPUs of its GPU\'s NUMA node')
    ap.add_argument('--gru-mode', type=int, default=0, help='debug: 0 auto, 1 CUDA-core, 2 mma.sync, 3 tcgen05, 7 mma.sync with 32-stream tiles')
    ap.add_argument('--k1-mode', type=int, default=0, help='debug (A/B runs only): 0 default MFCC kernel choice, 2 FFT kernel, 3 FFT kernel with 64-bit set-up, 4 tcgen05 stage 2 only, 5 both DFT stages on tcgen05')
    ap.add_argument('--dump-outputs', metavar='DIR', help='after the timed steps write what the last one returned (rank 0\'s streams) as DIR/<name>.npy: '
                    'raw, conf, fired, stream (the stream index of each row; a seeded sample above %d streams) and detections' % DUMP_MAX_STREAMS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs:
        if args.impl != 'b200':
            ap.error('--dump-outputs writes the outputs of the b200 arm')
        os.makedirs(args.dump_outputs, exist_ok=True)
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == 'reference':
        run_reference(args, int(os.environ.get('RANK', '0')))
        return
    run_b200(args)


if __name__ == '__main__':
    main()
