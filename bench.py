#!/usr/bin/env python
"""bench.py — encode->decode throughput of the colour-modem hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload pald576|ntsc3d600|sweep1080] [--frames F] [--dump-outputs DIR]

Workloads
  pald576    (default; BASELINE configs[1], the configuration the metric is quoted on): standard 625-line PAL, PAL-D
             decoder, 720x576.  A *step* is one pass of the hot path over one batch of F synthetic frames per GPU
             (default 8192: 20 steps keep the chip busy for ~2 s, so clocks and power reach their steady state):
                 composite = encode(rgb)        k_qam_encode_row
                 rgb'      = decode(composite)  k_qam_bs_row (2 field-top rows per frame) + k_qam_rows2<PALD> (all the
                                                filtering, one row per CTA) + k_qam_combine (pairing of neighbouring rows)
             Frames are sharded over ranks in contiguous ranges (rank r owns absolute frames [r*F, (r+1)*F)); no
             inter-GPU traffic (SURVEY.md §8e): "scaling": "weak".
  ntsc3d600  (BASELINE configs[2]): Simple3DCombModem(NtscCombModem) over a 600-frame 720x480 sequence cut into G contiguous
             frame ranges, one per GPU: "scaling": "strong" (total work fixed).
  sweep1080  (BASELINE configs[4]): the 16 preset / line-standard pairs on a 500-frame 1920x1080 batch, the frames of every
             preset cut into G ranges; a step is one pass over all presets.

`value` is whole-job frames/s with the batch resident in HBM (CUDA events, max over ranks); `e2e` is the same metric through
the public host API with pinned HOST buffers, every copy inside the timed region: ImageModem.transcode_batch
(cm_transcode_frames_host: RGB frames in, the decoded RGB frames out, the composite staying in device memory;
`e2e.with_composite_out` is the same call also copying the composite out), and beside it `e2e.two_calls`, the reference's two calls
ImageModem.modulate_batch / demodulate_batch (cm_encode_frames_host / cm_decode_frames_host) with the composite crossing the
link both ways.  After the timed region one frame of the timed batch is checked
against the float64 oracle; a difference above 1 LSB fails the run (exit code 3).

`--impl reference` times the CPU restatement of the reference (oracle/, float64 numpy/scipy — the reference is pure
Python and cannot travel to the GPU box) on all host cores, on a bounded sample of the same workload.
"""
import argparse
import json
import os
import queue
import re
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

W, H = 720, 576
METRIC = 'enc->dec frames/s at 576i (PalDModem PAL 720x576)'
BYTES_PER_FRAME = 3 * W * H + W * H + W * H + 3 * W * H          # SURVEY.md §8d: 3,317,760 B
DECODE_BYTES_PER_FRAME = W * H + 3 * W * H                        # composite in + RGB out of the decode kernels
# SURVEY.md §8d, measured on the reference (dense multiply-adds per pixel, encode + decode): PAL-D 10 + 430
MAC_PER_PIXEL = {'pald576': 440.0, 'ntsc3d600': 223.0}
ROWS_MAC_PER_PIXEL = 430.0 - 30.0       # pass 1 carries the decode chain except the pairing / re-modulation of pass 2


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--frames', type=int, default=0, help='frames per GPU per step (0 = the workload\'s default)')
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='pald576', choices=['pald576', 'ntsc3d600', 'sweep1080'])
    ap.add_argument('--cpu-frames', type=int, default=0, help='frames per worker in the CPU sample (0 = 8)')
    ap.add_argument('--e2e-frames', type=int, default=512, help='frames per host batch of the end-to-end measurement')
    ap.add_argument('--e2e-seconds', type=float, default=1.5, help='target length of each end-to-end timed region')
    ap.add_argument('--no-extras', action='store_true', help='skip the short runs of the other BASELINE configs')
    ap.add_argument('--no-cpu', action='store_true', help='skip the CPU baseline beside the GPU number')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write what the last timed step computed (rank 0) as DIR/<name>.npy in float32, a fixed seeded '
                         'sample of its rows of at most 64 MB, so that two builds can be compared output for output')
    a = ap.parse_args()
    if a.dump_outputs and a.impl != 'ours':
        ap.error('--dump-outputs needs --impl ours (the reference arm keeps no frames)')
    return a


# ------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port on all host cores
# ------------------------------------------------------------------------------------------------------------
_worker = {}


def _cpu_spec(workload):
    import oracle
    if workload == 'ntsc3d600':
        return oracle.ModemSpec('ntsc_3d', 'NTSC', 720, 480), 480, 720
    return oracle.ModemSpec('pal_d', 'PAL', W, H), H, W


def _cpu_init(workload):
    os.environ['OMP_NUM_THREADS'] = '1'
    import oracle
    spec, hh, ww = _cpu_spec(workload)
    _worker['modem'] = oracle.build(spec)
    _worker['size'] = (hh, ww)


def _cpu_range(rng):
    """encode->decode of the contiguous frame range [lo, hi) on one core.  Synthesising a frame is not timed (the GPU
    arm's inputs are resident before its timed region too).  Returns the seconds spent in encode->decode."""
    from oracle import frame as oframe
    from color_modem_b200.synth import synth_frames_u8
    lo, hi = rng
    hh, ww = _worker['size']
    acc, busy = 0, 0.0
    for i in range(lo, hi):
        rgb = synth_frames_u8(1, hh, ww, first_frame=i, seed=0)[0]       # (one frame at a time: the generator's int64
        t0 = time.perf_counter()                                        #  temporaries are 100 bytes per pixel)
        comp = oframe.encode_frame_u8(_worker['modem'], i, rgb)
        out = oframe.decode_frame_u8(_worker['modem'], i, comp)
        busy += time.perf_counter() - t0
        acc += int(out[0, 0, 0])
    return busy, acc


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_pool(workload):
    import multiprocessing as mp
    cores = host_cores()
    pool = mp.get_context('fork').Pool(cores, initializer=_cpu_init, initargs=(workload,))
    pool.map(_cpu_range, [(i, i + 1) for i in range(cores)], chunksize=1)     # untimed: spin up every worker, import scipy, design filters
    return pool, cores


def cpu_sample(pool, cores, nframes, first=0):
    """ONE map, one contiguous frame range per worker, no barrier inside.  Throughput = frames / the slowest worker's
    encode->decode time (inputs resident, like the GPU arm's `value`); also returns the wall time of the map (which
    includes synthesising the frames) and the summed CPU seconds."""
    bounds = [first + (k * nframes) // cores for k in range(cores + 1)]
    t0 = time.perf_counter()
    per = pool.map(_cpu_range, [(bounds[k], bounds[k + 1]) for k in range(cores)], chunksize=1)
    wall = time.perf_counter() - t0
    slowest = max(p[0] for p in per)
    return nframes / slowest, wall, sum(p[0] for p in per), slowest


def run_reference(args):
    if int(os.environ.get('RANK', '0')) != 0:
        return
    wl = args.workload if args.workload != 'sweep1080' else 'pald576'
    pool, cores = cpu_pool(wl)
    per_worker = args.cpu_frames or 8
    nframes = per_worker * cores                       # frames per step: a whole number per worker
    if args.warmup:
        cpu_sample(pool, cores, cores * min(args.warmup, 2))
    # all the steps as one map: a step is `nframes` frames, no barrier between steps
    fps, wall, cpu_s, slowest = cpu_sample(pool, cores, nframes * args.steps, first=0)
    pool.close()
    name = 'PalDModem PAL 720x576' if wl == 'pald576' else 'Simple3DCombModem(NtscCombModem) NTSC 720x480'
    line = {
        'impl': 'reference', 'metric': METRIC if wl == 'pald576' else 'enc->dec frames/s at 480i (%s)' % name,
        'value': fps, 'unit': 'frames/s', 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * slowest / max(args.steps, 1),
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': {'workload': '%s encode->decode; CPU oracle port (float64 numpy/scipy restatement of the reference, '
                               'vectorised over lines), %d frames per step over %d processes, all steps in one map'
                               % (name, nframes, cores)},
        'cpu_baseline': {'value': fps, 'unit': 'frames/s', 'cores': cores, 'kind': 'port',
                         'sample': '%d steps x %d frames of %s encode->decode, one contiguous frame range per core; slowest '
                                   'core %.1f s (the timed figure), %.1f s CPU in total, map wall %.1f s incl. frame synthesis'
                                   % (args.steps, nframes, name, slowest, cpu_s, wall)},
        'e2e': {'value': fps, 'unit': 'frames/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------------
class ClockSampler(object):
    QUERY = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
             'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
             'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index = index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.QUERY,
                                          '--format=csv,noheader,nounits', '-lms', '50'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append((time.perf_counter(), ln.strip()))

    def stop(self, t_begin, t_end):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        sm, power, smax, reasons = [], [], None, set()
        for t, ln in self.lines:
            if t < t_begin or t > t_end + 0.1:
                continue
            f = [x.strip() for x in ln.split(',')]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax = float(f[2])
                power.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[5:9]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        sm.sort()
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_min_mhz': sm[0] if sm else None, 'sm_max_mhz': smax,
                'power_w_max': max(power) if power else None, 'reasons': sorted(reasons), 'samples': len(sm),
                'covers_s': t_end - t_begin}


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            return float(json.load(f)['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    except Exception:
        return 6650.0, 'fallback (B200_PROFILING.md 6.65 TB/s)'


def fma_peak():
    import ctypes as C
    from color_modem_b200 import _native as N
    v = C.c_double(0.0)
    N.check(N.load().cm_measure_fma_peak(C.byref(v)))
    return v.value


def pcie_peak(torch, dev, nbytes=256 << 20, reps=6):
    """Bare pinned-memory copy ceiling of this rank's link: H2D alone, D2H alone, both directions at once (GB/s each way)."""
    h_in = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    h_out = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    d_a = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    d_b = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    s1, s2 = torch.cuda.Stream(dev), torch.cuda.Stream(dev)

    def run(up, down):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            if up:
                with torch.cuda.stream(s1):
                    d_a.copy_(h_in, non_blocking=True)
            if down:
                with torch.cuda.stream(s2):
                    h_out.copy_(d_b, non_blocking=True)
        torch.cuda.synchronize()
        return reps * nbytes / (time.perf_counter() - t0) / 1e9

    run(True, True)
    return {'h2d_gbs': run(True, False), 'd2h_gbs': run(False, True), 'both_each_way_gbs': run(True, True),
            'bytes_per_copy': nbytes}


def parity_check(kind, variant, hh, ww, frame, rgb, comp, out):
    """One frame of the timed batch against the float64 oracle (the checker, after the timing): max |difference| in LSB."""
    import numpy as np
    import oracle
    from oracle import frame as oframe
    om = oracle.build(oracle.ModemSpec(kind, variant, ww, hh))
    c_ref = oframe.encode_frame_u8(om, frame, rgb)
    o_ref = oframe.decode_frame_u8(om, frame, comp)
    return (int(np.abs(comp.astype(np.int32) - c_ref.astype(np.int32)).max()),
            int(np.abs(out.astype(np.int32) - o_ref.astype(np.int32)).max()))


class Dist(object):
    def __init__(self, torch):
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get('WORLD_SIZE', '1'))
        self.rank = int(os.environ.get('RANK', '0'))
        self.local = int(os.environ.get('LOCAL_RANK', '0'))
        if self.world > 1:
            os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
            dist.init_process_group('nccl', device_id=torch.device('cuda', self.local))
        torch.cuda.set_device(self.local)
        self.dev = torch.device('cuda', self.local)
        # host threads and pinned staging buffers of this rank on the NUMA node of its GPU (no-op where sysfs does not say)
        from color_modem_b200.shard import bind_to_gpu_numa_node
        self.numa_node = bind_to_gpu_numa_node(self.local)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max(self, v):
        t = self.torch.tensor([v], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum(self, v):
        t = self.torch.tensor([v], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return float(t.item())

    def close(self):
        if self.world > 1:
            self.dist.barrier()
            self.dist.destroy_process_group()


def timed_steps(D, step, steps, warmup):
    """W untimed steps, then exactly K steps bracketed by barrier + synchronize, CUDA events, max over ranks (ms)."""
    torch = D.torch
    for _ in range(warmup):
        step()
    D.barrier()
    t_begin = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    D.barrier()
    t_end = time.perf_counter()
    return D.max(e0.elapsed_time(e1)), t_begin, t_end


DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(dirname, first_frame, budget=DUMP_BYTES, prefix='', **arrays):
    """DIR/<prefix><name>.npy (float32) for each device array [frames, rows, ...] of one step, all at the same rows: a
    seeded choice of its rows (the same for the same arguments) that fits `budget` bytes; DIR/<prefix>frame_index.npy and
    DIR/<prefix>row_index.npy (float64) say which, in absolute frame numbers."""
    import numpy as np
    import torch
    n, h = next(iter(arrays.values())).shape[:2]
    per_row = 16 + sum(4 * a[0, 0].numel() for a in arrays.values())
    k = min(n * h, (budget - 4096) // per_row)
    pick = np.sort(np.random.default_rng(0).choice(n * h, k, replace=False))
    os.makedirs(dirname, exist_ok=True)
    np.save(os.path.join(dirname, prefix + 'frame_index.npy'), (first_frame + pick // h).astype(np.float64))
    np.save(os.path.join(dirname, prefix + 'row_index.npy'), (pick % h).astype(np.float64))
    for name, a in arrays.items():
        sample = a.reshape(n * h, *a.shape[2:])[torch.from_numpy(pick).to(a.device)].cpu().numpy()
        np.save(os.path.join(dirname, prefix + name + '.npy'), sample.astype(np.float32))


def tiled_frames(torch, dev, n, hh, ww, first_frame, seed=0, distinct=16):
    """[n, hh, ww, 3] u8 on the device: `distinct` synthetic frames tiled (content does not affect the data-independent
    kernels); returns (device tensor, numpy base)."""
    from color_modem_b200.synth import synth_frames_u8
    base = synth_frames_u8(min(n, distinct), hh, ww, first_frame=first_frame, seed=seed)
    reps = -(-n // base.shape[0])
    return torch.from_numpy(base).to(dev).repeat(reps, 1, 1, 1)[:n].contiguous(), base


def e2e_measure(D, args, make_modem, first_frame, hh, ww):
    """End to end through ImageModem on pinned host buffers.  Three figures, every byte copied inside the timed region:
      sequential  modulate_batch then demodulate_batch, one after the other, one thread
      pipelined   (headline) two host threads: the demodulation of batch i runs while batch i+1 is modulated, the composite
                  batches passed through a small ring of host buffers — a streaming user of the two reference calls
      transcode   ImageModem.transcode_batch: one call, the composite handed over in device memory (and still copied out)
      transcode_rgb  (headline) the same call with want_composite=False: RGB frames in, decoded RGB frames out — the result
                  of the encode->decode step of the metric; 3 + 3 bytes per pixel over the link"""
    torch = D.torch
    import numpy as np
    from color_modem_b200.image import ImageModem
    from color_modem_b200.synth import synth_frames_u8
    F = args.e2e_frames
    m1, m2 = make_modem(), make_modem()
    img, img2 = ImageModem(m1), ImageModem(m2)
    wc, wo = m1.composite_width, m1.output_width
    base = synth_frames_u8(min(F, 16), hh, ww, first_frame=first_frame, seed=0)
    host_rgb = torch.from_numpy(base).repeat(-(-F // base.shape[0]), 1, 1, 1)[:F].contiguous().pin_memory()
    ring = [torch.empty((F, hh, wc), dtype=torch.uint8).pin_memory() for _ in range(3)]
    host_out = torch.empty((F, hh, wo, 3), dtype=torch.uint8).pin_memory()
    np_rgb, np_out = host_rgb.numpy(), host_out.numpy()
    np_ring = [r.numpy() for r in ring]

    def sequential(n):
        for _ in range(n):
            img.modulate_batch(np_rgb, first_frame, out=np_ring[0])
            img.demodulate_batch(np_ring[0], first_frame, out=np_out)

    def pipelined(n):
        free, ready = queue.Queue(), queue.Queue()
        for b in range(len(np_ring)):
            free.put(b)
        err = []

        def producer():
            try:
                for _ in range(n):
                    b = free.get()
                    img.modulate_batch(np_rgb, first_frame, out=np_ring[b])
                    ready.put(b)
            except Exception as e:                                   # noqa: BLE001
                err.append(e)
                ready.put(None)

        th = threading.Thread(target=producer)
        th.start()
        for _ in range(n):
            b = ready.get()
            if b is None:
                break
            img2.demodulate_batch(np_ring[b], first_frame, out=np_out)
            free.put(b)
        th.join()
        if err:
            raise err[0]

    def transcode(n):
        for _ in range(n):
            img.transcode_batch(np_rgb, first_frame, out=np_out, comp_out=np_ring[0])

    def transcode_rgb(n):
        for _ in range(n):
            img.transcode_batch(np_rgb, first_frame, out=np_out, want_composite=False)

    def timed(fn, n):
        D.barrier()
        t0 = time.perf_counter()
        fn(n)
        D.barrier()
        return D.max(time.perf_counter() - t0)

    res = {}
    for name, fn in (('sequential', sequential), ('transcode', transcode), ('transcode_rgb', transcode_rgb),
                     ('pipelined', pipelined)):
        fn(2)                                                          # warm-up: handles, staging buffers, pipeline fill
        probe = timed(fn, 4) / 4
        n = max(4, min(400, int(args.e2e_seconds / max(probe, 1e-4))))
        n = int(D.max(n))
        res[name] = {'frames_per_s': F * D.world * n / timed(fn, n), 'steps': n}
    np_comp = np.array(np_ring[0][:1])       # (the transcode pass ran last on ring[0] before pipelined; any slot holds the batch)
    return res, np_rgb, np_ring, np_out, np_comp


def run_pald(args, D, cpu_line):
    torch = D.torch
    from color_modem_b200 import _native as N
    from color_modem_b200.line import LineConfig
    from color_modem_b200.color.pal import PalDModem

    F = args.frames or 8192
    first_frame = D.rank * F                      # contiguous frame range of this rank
    make = lambda: PalDModem(LineConfig((W, H)))  # noqa: E731
    modem = make()
    rgb, _ = tiled_frames(torch, D.dev, F, H, W, first_frame)
    comp = torch.empty((F, H, W), dtype=torch.uint8, device=D.dev)
    out = torch.empty((F, H, W, 3), dtype=torch.uint8, device=D.dev)

    def step():
        modem.encode_frames(rgb, first_frame=first_frame, out=comp)
        modem.decode_frames(comp, first_frame=first_frame, out=out)

    warmup = max(args.warmup, 3)
    sampler = ClockSampler(D.local)
    if D.rank == 0:
        sampler.start()
        time.sleep(0.2)
    launches0 = N.launch_count()
    ms, t_begin, t_end = timed_steps(D, step, args.steps, warmup)
    launches = (N.launch_count() - launches0) * args.steps // (args.steps + warmup)
    clocks = sampler.stop(t_begin, t_end) if D.rank == 0 else None
    if args.dump_outputs and D.rank == 0:
        dump_outputs(args.dump_outputs, first_frame, composite=comp, rgb=out)

    # ---- per-kernel device time (CUDA events around every launch), as run -----------------------------------------------
    modem.timing(True)
    D.barrier()
    ksteps = 3
    for _ in range(ksteps):
        step()
    D.barrier()
    k_ms = {name: modem.timing_read(kid) for name, kid in
            (('encode', N.K_ENCODE), ('bandsplit_top_rows', N.K_BANDSPLIT), ('pald_rows', N.K_PALD),
             ('combine', N.K_DECODE_OTHER))}
    modem.timing(False)
    # the same on a handle with the optional pass-1 / pass-2 overlap forced off: every kernel alone on the chip
    os.environ['CM_OVERLAP'] = '0'
    serial = make()
    serial._handle()
    del os.environ['CM_OVERLAP']
    serial.timing(True)
    for _ in range(2):
        serial.encode_frames(rgb, first_frame=first_frame, out=comp)
        serial.decode_frames(comp, first_frame=first_frame, out=out)
    D.barrier()
    k_serial = {name: serial.timing_read(kid) for name, kid in
                (('encode', N.K_ENCODE), ('bandsplit_top_rows', N.K_BANDSPLIT), ('pald_rows', N.K_PALD),
                 ('combine', N.K_DECODE_OTHER))}
    serial.timing(False)
    serial.close()

    # ---- parity gate: frame j of the timed batch against the oracle -----------------------------------------------------
    parity = None
    j = 7 % F
    if D.rank == 0:
        lsb_c, lsb_o = parity_check('pal_d', 'PAL', H, W, first_frame + j, rgb[j].cpu().numpy(), comp[j].cpu().numpy(),
                                    out[j].cpu().numpy())
        parity = {'frame': first_frame + j, 'max_lsb_comp': lsb_c, 'max_lsb_rgb': lsb_o,
                  'checker': 'float64 oracle (oracle/), whole 720x576 frame of the timed batch, after the timing'}
    del rgb, comp, out
    torch.cuda.empty_cache()

    # ---- end to end ---------------------------------------------------------------------------------------------------------
    link = pcie_peak(torch, D.dev)
    e2e, np_rgb, np_ring, np_out, _ = e2e_measure(D, args, make, first_frame, H, W)
    if D.rank == 0:
        lsb_c, lsb_o = parity_check('pal_d', 'PAL', H, W, first_frame + j, np_rgb[j], np_ring[0][j], np_out[j])
        parity['e2e_max_lsb_comp'], parity['e2e_max_lsb_rgb'] = lsb_c, lsb_o
    link_min = D.max(-link['both_each_way_gbs'])
    Fe = args.e2e_frames
    h2d, d2h = Fe * (3 * W * H + W * H), Fe * (W * H + 3 * W * H)

    others = []
    if not args.no_extras:
        others = other_workloads(D)

    if D.rank == 0:
        fps = F * D.world * args.steps / (ms * 1e-3)
        peak, peak_src = measured_peak_gbs()
        tfma = fma_peak()
        step_ms = ms / args.steps

        def per_launch(d, key):
            t, n = d[key]
            return t / max(n, 1), n

        rows_ms, rows_n = per_launch(k_ms, 'pald_rows')
        rows_serial_ms, rows_serial_n = per_launch(k_serial, 'pald_rows')
        fpl = F * ksteps / max(rows_n, 1)                       # frames per launch
        fpl_serial = F * 2 / max(rows_serial_n, 1)
        achieved = fpl * DECODE_BYTES_PER_FRAME / (rows_ms * 1e-3) / 1e9 if rows_ms > 0 else 0.0
        achieved_serial = fpl_serial * DECODE_BYTES_PER_FRAME / (rows_serial_ms * 1e-3) / 1e9 if rows_serial_ms > 0 else 0.0
        traffic = None
        try:
            with open(os.path.join(ROOT, 'profiles', 'r2_traffic.json')) as tf:
                traffic = json.load(tf)
        except Exception:
            pass
        ksum = {k: v[0] / ksteps for k, v in k_ms.items()}
        ksum_serial = {k: v[0] / 2 for k, v in k_serial.items()}
        px_s = fps / D.world * W * H
        rows_px_s = fpl_serial * W * H / (rows_serial_ms * 1e-3) if rows_serial_ms > 0 else 0.0
        line = {
            'metric': METRIC, 'value': fps, 'unit': 'frames/s', 'n_gpus': D.world, 'steps': args.steps,
            'warmup': warmup, 'ms_per_step': step_ms, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': 'PalDModem PAL 720x576 encode->decode (BASELINE configs[1])',
                       'frames_per_gpu_per_step': F, 'sharding': 'contiguous frame ranges, no inter-GPU traffic',
                       'timed_region_s': ms * 1e-3,
                       'l2': 'no flush: each step streams %.1f GB per GPU (>> 126 MB L2)' % (F * BYTES_PER_FRAME / 1e9)},
            'clocks': clocks,
            'parity': parity,
            'e2e': {'value': e2e['transcode_rgb']['frames_per_s'], 'unit': 'frames/s',
                    'h2d_bytes_per_step': Fe * 3 * W * H, 'd2h_bytes_per_step': Fe * 3 * W * H, 'frames_per_step': Fe,
                    'steps': e2e['transcode_rgb']['steps'],
                    'api': 'ImageModem.transcode_batch(want_composite=False) (cm_transcode_frames_host) on pinned host buffers: RGB '
                           'frames in, the decoded RGB frames of the encode->decode step out, the composite handed from the encoder '
                           'to the decoder in device memory; every copy inside the timed region',
                    'with_composite_out': {'value': e2e['transcode']['frames_per_s'], 'steps': e2e['transcode']['steps'],
                                           'h2d_bytes_per_step': Fe * 3 * W * H, 'd2h_bytes_per_step': d2h,
                                           'api': 'the same call also copying the composite frames out (what the reference '
                                                  'cli.py:62-65 can save): 3 bytes per pixel in, 4 out',
                                           'frac_of_copy_peak': e2e['transcode']['frames_per_s'] / D.world * (d2h / Fe) / 1e9
                                           / (-link_min)},
                    'two_calls': {'value': e2e['pipelined']['frames_per_s'], 'steps': e2e['pipelined']['steps'],
                                  'api': 'ImageModem.modulate_batch then demodulate_batch (cm_encode_frames_host / '
                                         'cm_decode_frames_host), the composite through host memory both ways; two host threads, '
                                         'batch i demodulated while batch i+1 is modulated, composites through a ring of 3 host '
                                         'buffers',
                                  'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
                                  'sequential': e2e['sequential']['frames_per_s'],
                                  'frac_of_copy_peak': e2e['pipelined']['frames_per_s'] / D.world * (h2d / Fe) / 1e9 / (-link_min)},
                    'numa_node_of_rank0': D.numa_node,
                    'copy_peak': dict(link, min_over_ranks_both_each_way_gbs=-link_min,
                                      how='bare pinned cudaMemcpyAsync of 256 MiB, H2D alone / D2H alone / both at once'),
                    'achieved_d2h_gbs': e2e['transcode_rgb']['frames_per_s'] / D.world * 3 * W * H / 1e9,
                    'frac_of_copy_peak': e2e['transcode_rgb']['frames_per_s'] / D.world * 3 * W * H / 1e9 / (-link_min),
                    'frac_note': 'bytes per second of one direction (3 B/pixel each way) over the measured ceiling of one '
                                 'direction while both are busy'},
            'gpu_launches': launches,
            'other_workloads': others,
            'roofline': {'bound': 'hbm', 'kernel': 'k_qam_rows2<float, PALD, 1>', 'achieved': achieved, 'peak': peak,
                         'unit': 'GB/s', 'frac': achieved / peak,
                         'traffic': (traffic['k_qam_rows2']['dram_bytes_per_launch'] * fpl
                                     / traffic['k_qam_rows2']['frames_per_launch']) if traffic else None,
                         'traffic_source': traffic['source'] if traffic else None,
                         'peak_source': peak_src,
                         'algorithmic_bytes_per_launch': fpl * DECODE_BYTES_PER_FRAME,
                         'frames_per_launch': fpl, 'avg_launch_ms': rows_ms,
                         'timing': 'CUDA events on the launch stream around every launch of the kernel, over %d steps run '
                                   'right after the timed region (same buffers, same launches)' % ksteps,
                         'alone_on_the_chip': {'avg_launch_ms': rows_serial_ms, 'frames_per_launch': fpl_serial,
                                               'achieved': achieved_serial, 'frac': achieved_serial / peak},
                         'kernel_ms_per_step': ksum, 'kernel_ms_per_step_serial': ksum_serial,
                         'kernel_share_of_step_serial': {k: v / max(sum(ksum_serial.values()), 1e-9)
                                                         for k, v in ksum_serial.items()},
                         'whole_chain_frac': fps / D.world * BYTES_PER_FRAME / 1e9 / peak,
                         'note': 'the decode chain is bound by instruction issue and the FP32 pipe, not by HBM: see '
                                 'roofline_fma and profiles/r2_pald_summary.md'},
            'roofline_fma': {'bound': 'fp32 multiply-add', 'peak': tfma, 'unit': 'TFMA/s',
                             'peak_source': 'measured live (cm_measure_fma_peak: packed FFMA2, uniform operands, all SMs)',
                             'mac_per_pixel': MAC_PER_PIXEL['pald576'],
                             'mac_source': 'SURVEY.md §8d: dense multiply-adds per pixel of the reference chain, encode 10 + '
                                           'decode 430 (half-band zero taps included)',
                             'achieved': px_s * MAC_PER_PIXEL['pald576'] / 1e12,
                             'frac': px_s * MAC_PER_PIXEL['pald576'] / 1e12 / tfma,
                             'dominant_kernel': {'kernel': 'k_qam_rows2<float, PALD, 1>', 'mac_per_pixel': ROWS_MAC_PER_PIXEL,
                                                 'achieved': rows_px_s * ROWS_MAC_PER_PIXEL / 1e12,
                                                 'frac': rows_px_s * ROWS_MAC_PER_PIXEL / 1e12 / tfma}},
        }
        if cpu_line is not None:
            line['cpu_baseline'] = cpu_line
        print(json.dumps(line), flush=True)
        bad = max(parity['max_lsb_comp'], parity['max_lsb_rgb'], parity['e2e_max_lsb_comp'], parity['e2e_max_lsb_rgb'])
        return 3 if bad > 1 else 0
    return 0


def other_workloads(D):
    """The other BASELINE configs, briefly (device-resident, CUDA events, max over ranks): context for the headline."""
    torch = D.torch
    from color_modem_b200 import comb
    from color_modem_b200.color import ntsc, secam, niir
    from color_modem_b200.line import LineConfig
    from color_modem_b200.shard import frame_range
    others = []
    lc480 = LineConfig((720, 480))
    # configs[2]: 600 NTSC frames cut into one contiguous range per GPU — strong scaling
    lo, hi = frame_range(600, D.rank, D.world)
    mm = comb.Simple3DCombModem(ntsc.NtscCombModem(lc480))
    xr, _ = tiled_frames(torch, D.dev, hi - lo, 480, 720, lo, seed=2, distinct=8)
    xc = mm.encode_frames(xr, first_frame=lo)
    xo = mm.decode_frames(xc, first_frame=lo)

    def step():
        mm.encode_frames(xr, first_frame=lo, out=xc)
        mm.decode_frames(xc, first_frame=lo, out=xo)

    reps = 20
    ms, _, _ = timed_steps(D, step, reps, 3)
    fps = 600 * reps / (ms * 1e-3)
    bytes_x = 3 * 720 * 480 + 2 * 720 * 480 + 3 * 720 * 480
    others.append({'workload': 'Simple3DCombModem(NtscCombModem) NTSC 720x480, 600-frame sequence in %d contiguous frame '
                               'range(s) (BASELINE configs[2], north_star 480i target)' % D.world,
                   'scaling': 'strong', 'frames_per_s': fps, 'frames_per_gpu': hi - lo, 'n_gpus': D.world,
                   'hbm_roofline_frac': fps / D.world * bytes_x / 1e9 / measured_peak_gbs()[0]})
    del mm, xr, xc, xo
    if D.rank == 0:
        extra = [('NtscModem NTSC 720x480 (BASELINE configs[0])', lambda: ntsc.NtscModem(lc480), 480, 256),
                 ('ColorAveragingModem(SecamModem) SECAM 720x576 x 1000 frames (BASELINE configs[3])',
                  lambda: comb.ColorAveragingModem(secam.SecamModem(LineConfig((W, H)))), H, 1000),
                 ('HueCorrectingNiirModem 720x576 x 1000 frames (BASELINE configs[3])',
                  lambda: niir.HueCorrectingNiirModem(LineConfig((W, H))), H, 1000)]
        for name, make, hh, fr in extra:
            mm = make()
            xr, _ = tiled_frames(torch, D.dev, fr, hh, W, 0, seed=2, distinct=8)
            xc = mm.encode_frames(xr)
            xo = mm.decode_frames(xc)
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(5):
                mm.encode_frames(xr, out=xc)
                mm.decode_frames(xc, out=xo)
            b.record()
            torch.cuda.synchronize()
            fps_x = 5 * fr / (a.elapsed_time(b) * 1e-3)
            bytes_x = 3 * W * hh + 2 * mm.composite_width * hh + 3 * mm.output_width * hh
            others.append({'workload': name, 'frames_per_s': fps_x, 'frames_per_step': fr, 'n_gpus': 1,
                           'hbm_roofline_frac': fps_x * bytes_x / 1e9 / measured_peak_gbs()[0]})
            del mm, xr, xc, xo
    if D.world > 1:
        D.dist.barrier()
    return others


def run_ntsc3d600(args, D, cpu_line):
    """BASELINE configs[2]: strong scaling of a 600-frame sequence (override with --frames)."""
    torch = D.torch
    from color_modem_b200 import _native as N
    from color_modem_b200 import comb
    from color_modem_b200.color import ntsc
    from color_modem_b200.line import LineConfig
    from color_modem_b200.shard import frame_range
    total = args.frames or 600
    lo, hi = frame_range(total, D.rank, D.world)
    hh, ww = 480, 720
    modem = comb.Simple3DCombModem(ntsc.NtscCombModem(LineConfig((ww, hh))))
    rgb, _ = tiled_frames(torch, D.dev, hi - lo, hh, ww, lo, distinct=8)
    comp = modem.encode_frames(rgb, first_frame=lo)
    out = modem.decode_frames(comp, first_frame=lo)

    def step():
        modem.encode_frames(rgb, first_frame=lo, out=comp)
        modem.decode_frames(comp, first_frame=lo, out=out)

    warmup = max(args.warmup, 3)
    sampler = ClockSampler(D.local)
    if D.rank == 0:
        sampler.start()
        time.sleep(0.2)
    launches0 = N.launch_count()
    ms, t_begin, t_end = timed_steps(D, step, args.steps, warmup)
    launches = (N.launch_count() - launches0) * args.steps // (args.steps + warmup)
    clocks = sampler.stop(t_begin, t_end) if D.rank == 0 else None
    if args.dump_outputs and D.rank == 0:
        dump_outputs(args.dump_outputs, lo, composite=comp, rgb=out)
    if D.rank == 0:
        j = min(3, hi - lo - 1)
        lsb_c, lsb_o = parity_check('ntsc_3d', 'NTSC', hh, ww, lo + j, rgb[j].cpu().numpy(), comp[j].cpu().numpy(),
                                    out[j].cpu().numpy())
        fps = total * args.steps / (ms * 1e-3)
        bpf = 3 * ww * hh + 2 * ww * hh + 3 * ww * hh
        peak, peak_src = measured_peak_gbs()
        tfma = fma_peak()
        line = {'metric': 'enc->dec frames/s at 480i (Simple3DCombModem(NtscCombModem) NTSC 720x480)', 'value': fps,
                'unit': 'frames/s', 'n_gpus': D.world, 'steps': args.steps, 'warmup': warmup,
                'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None,
                'dtype': 'f32', 'data': 'synthetic',
                'config': {'workload': 'Simple3DCombModem(NtscCombModem) NTSC 720x480, %d-frame sequence in %d contiguous '
                                       'frame ranges (BASELINE configs[2])' % (total, D.world),
                           'frames_per_gpu_per_step': hi - lo, 'timed_region_s': ms * 1e-3,
                           'l2': 'each step streams %.0f MB per GPU' % ((hi - lo) * bpf / 1e6)},
                'clocks': clocks, 'gpu_launches': launches,
                'parity': {'frame': lo + j, 'max_lsb_comp': lsb_c, 'max_lsb_rgb': lsb_o},
                'roofline': {'bound': 'hbm', 'achieved': fps / D.world * bpf / 1e9, 'peak': peak, 'unit': 'GB/s',
                             'frac': fps / D.world * bpf / 1e9 / peak, 'traffic': None, 'peak_source': peak_src,
                             'kernel': 'whole chain (encode + k_qam_rows2<STD> + k_qam_combine<NTSC3>)'},
                'roofline_fma': {'peak': tfma, 'unit': 'TFMA/s', 'mac_per_pixel': MAC_PER_PIXEL['ntsc3d600'],
                                 'achieved': fps / D.world * ww * hh * MAC_PER_PIXEL['ntsc3d600'] / 1e12,
                                 'frac': fps / D.world * ww * hh * MAC_PER_PIXEL['ntsc3d600'] / 1e12 / tfma}}
        if cpu_line is not None:
            line['cpu_baseline'] = cpu_line
        print(json.dumps(line), flush=True)
        return 3 if max(lsb_c, lsb_o) > 1 else 0
    return 0


def run_sweep1080(args, D, cpu_line):
    """BASELINE configs[4]: every preset on a 500-frame 1920x1080 batch, frames of each preset cut into one range per GPU."""
    torch = D.torch
    from color_modem_b200 import _native as N
    from color_modem_b200.shard import frame_range
    sys.path.insert(0, os.path.join(ROOT, 'tools'))
    import sweep
    total = args.frames or 500
    lo, hi = frame_range(total, D.rank, D.world)
    hh, ww = 1080, 1920
    cases = sweep.hd_cases()
    modems = [(name, make()) for name, make in cases]
    rgb, _ = tiled_frames(torch, D.dev, hi - lo, hh, ww, lo, distinct=4)
    bufs = {}
    for name, m in modems:
        key = (m.composite_width, m.output_width)
        if key not in bufs:
            bufs[key] = (torch.empty((hi - lo, hh, key[0]), dtype=torch.uint8, device=D.dev),
                         torch.empty((hi - lo, hh, key[1], 3), dtype=torch.uint8, device=D.dev))
    per = {name: [torch.cuda.Event(enable_timing=True) for _ in range(2)] for name, _ in modems}

    def step(record=False):
        for name, m in modems:
            c, o = bufs[(m.composite_width, m.output_width)]
            if record:
                per[name][0].record()
            m.encode_frames(rgb, first_frame=lo, out=c)
            m.decode_frames(c, first_frame=lo, out=o)
            if record:
                per[name][1].record()

    warmup = max(args.warmup, 3)
    sampler = ClockSampler(D.local)
    if D.rank == 0:
        sampler.start()
        time.sleep(0.2)
    launches0 = N.launch_count()
    ms, t_begin, t_end = timed_steps(D, step, args.steps, warmup)
    launches = (N.launch_count() - launches0) * args.steps // (args.steps + warmup)
    clocks = sampler.stop(t_begin, t_end) if D.rank == 0 else None
    if args.dump_outputs and D.rank == 0:
        # presets share output buffers, so each one's pass of the timed step is replayed and written before the next
        for name, m in modems:
            c, o = bufs[(m.composite_width, m.output_width)]
            m.encode_frames(rgb, first_frame=lo, out=c)
            m.decode_frames(c, first_frame=lo, out=o)
            dump_outputs(args.dump_outputs, lo, DUMP_BYTES // len(modems), re.sub(r'[^A-Za-z0-9]+', '_', name) + '.',
                         composite=c, rgb=o)
    step(record=True)
    D.barrier()
    rows = []
    for name, m in modems:
        t = D.max(per[name][0].elapsed_time(per[name][1]))
        rows.append({'modem': name, 'frames_per_s': total / (t * 1e-3), 'us_per_frame_per_gpu': 1e3 * t / (hi - lo)})
    if D.rank == 0:
        fps = total * len(modems) * args.steps / (ms * 1e-3)
        bpf = 3 * ww * hh + 2 * ww * hh + 3 * ww * hh
        peak, peak_src = measured_peak_gbs()
        line = {'metric': 'enc->dec frames/s, 1920x1080 sweep over %d presets' % len(modems), 'value': fps,
                'unit': 'frames/s', 'n_gpus': D.world, 'steps': args.steps, 'warmup': warmup,
                'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None,
                'dtype': 'f32', 'data': 'synthetic',
                'config': {'workload': 'all %d preset / line-standard pairs of BASELINE configs[4] on a %d-frame 1920x1080 '
                                       'batch, frames of every preset in %d contiguous ranges; a step is one pass over all '
                                       'presets' % (len(modems), total, D.world),
                           'frames_per_gpu_per_step': (hi - lo) * len(modems), 'timed_region_s': ms * 1e-3,
                           'l2': 'each preset pass streams %.1f GB per GPU' % ((hi - lo) * bpf / 1e9)},
                'clocks': clocks, 'gpu_launches': launches, 'presets': rows,
                'roofline': {'bound': 'hbm', 'achieved': fps / D.world * bpf / 1e9, 'peak': peak, 'unit': 'GB/s',
                             'frac': fps / D.world * bpf / 1e9 / peak, 'traffic': None, 'peak_source': peak_src,
                             'kernel': 'whole chain, mean over the presets'}}
        print(json.dumps(line), flush=True)
    return 0


def run_ours(args):
    rank = int(os.environ.get('RANK', '0'))
    cpu_line = None
    if rank == 0 and not args.no_cpu and args.workload != 'sweep1080':
        # CPU baseline beside the GPU number: oracle port on all host cores, bounded sample.  Taken before CUDA is
        # initialised so the worker processes can be forked safely.
        pool, cores = cpu_pool(args.workload)
        nfr = (args.cpu_frames or 8) * cores
        cfps, wall, cpu_s, slowest = cpu_sample(pool, cores, nfr)
        pool.close()
        pool.join()
        what = '720x576 PAL-D' if args.workload == 'pald576' else '720x480 NTSC 3-line comb'
        cpu_line = {'value': cfps, 'unit': 'frames/s', 'cores': cores, 'kind': 'port',
                    'sample': '%d frames of %s encode->decode through the float64 oracle port, one contiguous frame range per '
                              'core on %d cores; slowest core %.1f s (the timed figure), %.1f s CPU in total'
                              % (nfr, what, cores, slowest, cpu_s)}
    import torch
    D = Dist(torch)
    rc = {'pald576': run_pald, 'ntsc3d600': run_ntsc3d600, 'sweep1080': run_sweep1080}[args.workload](args, D, cpu_line)
    D.close()
    return rc


def main():
    args = parse()
    if args.impl == 'reference':
        run_reference(args)
        return 0
    return run_ours(args)


if __name__ == '__main__':
    sys.exit(main())
