"""End-to-end rate of ImageModem.transcode_batch with rgb24 and with yuv420p pictures on pinned host buffers (PAL-D 720x576,
the same pictures in both arms), and the device time of the two conversion kernels.  One JSON line:

    python tools/e2e_pixfmt.py [--frames 2048] [--seconds 1.5] [--rounds 2] [--trace DIR]

* the card's name and power limit (nvidia-smi, read-only) and the pinned two-way copy ceiling (bench.pcie_peak);
* transcode_batch rgb24 vs yuv420p (BT.601 limited), alternated A/B/A/B, calls of --frames frames, each arm timed for at
  least --seconds; the composite stays on the device (want_composite=False), as in bench.py's e2e headline;
* each conversion kernel timed with CUDA events on a 512-frame batch (318 MB of yuv420p, 637 MB of RGB: above the 126 MB L2),
  its achieved GB/s (bytes read + written) beside a device-to-device copy of 1 GiB measured the same way;
* after the timing: the yuv420p output must equal from_rgb24 of the rgb24 output.
--trace DIR also writes a torch.profiler trace of one yuv420p call (a run of its own, after everything else) and a summary of
the busy time of each stream."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch                                                            # noqa: E402
import bench                                                            # noqa: E402
from color_modem_b200.line import LineConfig                             # noqa: E402
from color_modem_b200.color.pal import PalDModem                         # noqa: E402
from color_modem_b200.image import ImageModem                            # noqa: E402
from color_modem_b200.pixfmt import PixelFormat, frame_bytes, from_rgb24, to_rgb24      # noqa: E402
from color_modem_b200.synth import synth_frames_u8                       # noqa: E402


def card():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [v.strip() for v in out.split(',')]
        return {'name': name, 'power_limit': power}
    except Exception as e:                                              # noqa: BLE001
        return {'name': 'unknown (%s)' % e, 'power_limit': 'unknown'}


def event_ms(fn, reps):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def stream_summary(trace_path):
    """Busy milliseconds of kernels and copies per CUDA stream in a chrome trace written by torch.profiler."""
    with open(trace_path) as f:
        events = json.load(f).get('traceEvents', [])
    per = {}
    for e in events:
        cat = e.get('cat', '')
        if cat not in ('kernel', 'gpu_memcpy') or 'dur' not in e:
            continue
        s = per.setdefault(str(e.get('args', {}).get('stream', e.get('tid'))), {'kernel_ms': 0.0, 'memcpy_ms': 0.0, 'n': 0,
                                                                               't0': e['ts'], 't1': e['ts'] + e['dur']})
        s['kernel_ms' if cat == 'kernel' else 'memcpy_ms'] += e['dur'] / 1e3
        s['n'] += 1
        s['t0'], s['t1'] = min(s['t0'], e['ts']), max(s['t1'], e['ts'] + e['dur'])
    for s in per.values():
        s['span_ms'] = (s.pop('t1') - s.pop('t0')) / 1e3
    return per


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--frames', type=int, default=2048)
    ap.add_argument('--seconds', type=float, default=1.5)
    ap.add_argument('--rounds', type=int, default=2)
    ap.add_argument('--trace', default=None)
    args = ap.parse_args()
    F, h, w = args.frames, 576, 720
    dev = torch.device('cuda', 0)
    fmt = PixelFormat('yuv420p', 'bt601', 'limited')
    fb = frame_bytes(fmt, w, h)
    res = {'metric': 'transcode_batch frames/s, PalDModem 720x576, pinned host buffers, rgb24 vs yuv420p', 'gpu': card(),
           'frames_per_call': F, 'pix_fmt': repr(fmt)}
    res['pcie'] = bench.pcie_peak(torch, dev)

    # the same pictures in both arms: yuv420p of the synthetic frames, and its rgb24 expansion
    base = torch.from_numpy(synth_frames_u8(16, h, w, seed=0)).to(dev)
    yuv16 = from_rgb24(base, fmt)
    rgb16 = to_rgb24(yuv16, fmt, w, h)
    reps = -(-F // 16)
    yuv = yuv16.cpu().repeat(reps, 1)[:F].contiguous().pin_memory().numpy()
    rgb = rgb16.cpu().repeat(reps, 1, 1, 1)[:F].contiguous().pin_memory().numpy()
    out_yuv = torch.empty((F, fb), dtype=torch.uint8).pin_memory().numpy()
    out_rgb = torch.empty((F, h, w, 3), dtype=torch.uint8).pin_memory().numpy()
    img = ImageModem(PalDModem(LineConfig((w, h))))
    arms = {'rgb24': lambda: img.transcode_batch(rgb, 0, out=out_rgb, want_composite=False),
            'yuv420p': lambda: img.transcode_batch(yuv, 0, out=out_yuv, want_composite=False, pix_fmt=fmt)}
    for fn in arms.values():
        fn()
        fn()
    runs = {k: [] for k in arms}
    for _ in range(args.rounds):
        for k, fn in arms.items():
            torch.cuda.synchronize()
            t0, n = time.perf_counter(), 0
            while n < 2 or time.perf_counter() - t0 < args.seconds:
                fn()
                n += 1
            runs[k].append(F * n / (time.perf_counter() - t0))
    link = res['pcie']['both_each_way_gbs']
    for k, v in runs.items():
        pb = fb if k == 'yuv420p' else 3 * w * h
        res[k] = {'frames_per_s': max(v), 'runs': v, 'link_bytes_per_frame_each_way': pb,
                  'achieved_each_way_gbs': max(v) * pb / 1e9, 'frac_of_copy_peak': max(v) * pb / 1e9 / link}
    res['speedup_yuv420p_over_rgb24'] = res['yuv420p']['frames_per_s'] / res['rgb24']['frames_per_s']

    # conversion kernels, device time, batches above L2
    n = 512
    d_yuv = yuv16.repeat(n // 16, 1).contiguous()
    d_rgb = torch.empty((n, h, w, 3), dtype=torch.uint8, device=dev)
    d_yuv2 = torch.empty_like(d_yuv)
    ms_to = event_ms(lambda: to_rgb24(d_yuv, fmt, w, h, out=d_rgb), 20)
    ms_from = event_ms(lambda: from_rgb24(d_rgb, fmt, out=d_yuv2), 20)
    big_a = torch.empty(1 << 30, dtype=torch.uint8, device=dev)
    big_b = torch.empty_like(big_a)
    ms_copy = event_ms(lambda: big_b.copy_(big_a), 10)
    copy_gbs = 2 * big_a.numel() / ms_copy / 1e6
    moved = n * (fb + 3 * w * h)
    res['kernels'] = {
        'frames': n, 'bytes_per_launch': moved,
        'hbm_copy_gbs_measured': copy_gbs,
        'k_yuv420p_to_rgb24': {'us_per_frame': ms_to * 1e3 / n, 'gbs': moved / ms_to / 1e6,
                               'frac_of_copy': moved / ms_to / 1e6 / copy_gbs},
        'k_rgb24_to_yuv420p': {'us_per_frame': ms_from * 1e3 / n, 'gbs': moved / ms_from / 1e6,
                               'frac_of_copy': moved / ms_from / 1e6 / copy_gbs},
    }
    del big_a, big_b

    # parity, after the timing: the yuv420p output is from_rgb24 of the rgb24 output, on the same pictures
    img.transcode_batch(rgb, 0, out=out_rgb, want_composite=False)
    img.transcode_batch(yuv, 0, out=out_yuv, want_composite=False, pix_fmt=fmt)
    ok = True
    for lo in range(0, F, 256):
        ref = from_rgb24(torch.from_numpy(out_rgb[lo:lo + 256]).to(dev), fmt).cpu().numpy()
        ok = ok and bool((ref == out_yuv[lo:lo + 256]).all())
    res['parity_yuv_equals_from_rgb24_of_rgb_path'] = ok

    if args.trace:
        from torch.profiler import ProfilerActivity, profile
        os.makedirs(args.trace, exist_ok=True)
        small = 256
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            img.transcode_batch(yuv[:small], 0, out=out_yuv[:small], want_composite=False, pix_fmt=fmt)
            torch.cuda.synchronize()
        path = os.path.join(args.trace, 'e2e_pixfmt_trace.json')
        prof.export_chrome_trace(path)
        res['trace'] = {'frames': small, 'streams': stream_summary(path)}
    print(json.dumps(res))
    if not ok:
        sys.exit(1)


if __name__ == '__main__':
    main()
