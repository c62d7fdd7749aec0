"""Time TableTennisPipeline.live against predict: S simulated cameras push synthetic 1080p frames (numpy, pageable memory) on a host
clock at a given fps, and each camera's 50-frame rallies end on schedule.

  latency : one camera at --fps; per rally, the time from the end_rally call to its result on the host (spin synchronised, positions
            already there), then predict on the same 50 frames at rally end, timed the same way; results compared bit for bit.
  k       : frames/s of one camera pushing as fast as it can (no clock), one frame per push, for several k (ready stacks per pass).
  max_fps : for S = 1, 2, 4 the largest per-camera fps of a ladder at which the pushes keep to the camera clock: the 95th percentile
            of (push returns - frame due) stays below one frame interval.  Rally ends are staggered over the cameras; the end_rally
            calls run on the same host thread, so their latency counts against the clock too.
With --devices N,M,...:
  launcher: (N = 1) devices=None against devices=[0] on one GPU: the max_fps arm for S = 1, 2, 4, with push p50 / p99.
  scaling : (N >= 2) devices=[0 .. N-1], one entry per GPU: the max_fps arm for S = 2, 4, 8, 16 cameras (S >= N), with end_rally median
            / p99.  An arm runs only where N GPUs are visible; the others, and S < N, are listed under 'skipped'.
--known-table: instead, the cameras arm: at --fps (default 30 here) the most cameras, of 1 .. 8, whose pushes keep to the clock, with
every stream's table set (LiveSession.set_table, the keypoints filtered from the pool's first 50 frames) against the tables detected,
with push p50 / p99 and end_rally median / p99 of every trial.
Pipelines (--pipeline): wasb-hrnet = WASB main + aux at 1280x704, HRNet main + aux (tf32), uplift (tf32x3) -- bench.py's pipeline leg;
default = the pipeline's default composition, ViTPose main (1152x640, tf32x3) + WASB aux for the ball, ViTPose main + HRNet aux for the
table.  The synthetic ViTPose and WASB ball detectors do not agree, so on `default` predict and end_rally refuse every rally with
ValueError after all detectors and filters have run (counted as 'refused'; latency then compares the two errors).  Writes one JSON file.

    python tools/time_live.py --out profiles/r06_live_timing.json
    python tools/time_live.py --out profiles/r07_live_devices_timing.json --pipeline default --devices 1,2,4,8
    python tools/time_live.py --out profiles/r10_known_table_live.json --known-table [--pipeline default]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), '..'))
from time_clips import write_checkpoints      # noqa: E402  (tools/ is the script's directory)

RALLY = 50
VIT_RES = (1152, 640)       # ViTPose input resolution, as in bench.py
LADDER = (30, 60, 90, 120, 150, 180, 240)


def write_vitpose_checkpoints(hub):
    """Ball and table ViTPose checkpoints beside write_checkpoints' WASB / HRNet / uplift ones (the default composition's main models)."""
    from upliftingtabletennis_b200 import synthetic, vitpose
    w = os.path.join(hub, 'checkpoints', 'tt_uplifting_extracted', 'weights')
    tokens = (VIT_RES[0] // 16) * (VIT_RES[1] // 16)
    for sub, sd, info in (
            ('inference_balldetection/vitpose', synthetic.vit_state_dict(vitpose.state_dict_layout(9, tokens, 1), seed=5),
             {'model_name': 'vitpose', 'image_resolution': VIT_RES, 'in_frames': 3, 'lr': 0.0}),
            ('inference_tabledetection/vitpose', synthetic.vit_state_dict(vitpose.state_dict_layout(3, tokens, 13), seed=6),
             {'model_name': 'vitpose', 'image_resolution': VIT_RES})):
        os.makedirs(os.path.join(w, sub), exist_ok=True)
        torch.save({'model_state_dict': sd, 'identifier': 'synthetic', 'additional_info': info}, os.path.join(w, sub, 'model.pt'))


def wait_until(t):
    d = t - time.perf_counter()
    if d > 0:
        time.sleep(d)


def outcome(fn):
    try:
        return fn()
    except ValueError:
        return ValueError


def latency(pipe, pool, fps, rallies):
    """One camera at fps: end_rally -> host result, and predict on the same rally at its end."""
    live_ms, predict_ms, same, refused = [], [], True, 0
    with pipe.live(fps) as live:
        for r in range(rallies + 1):                            # rally 0 warms up
            frames = [pool[(r * RALLY + j) % len(pool)] for j in range(RALLY)]
            t0 = time.perf_counter()
            for j, f in enumerate(frames):
                wait_until(t0 + j / fps)
                live.push(0, f)
            wait_until(t0 + RALLY / fps)
            t = time.perf_counter()
            got = outcome(lambda: live.end_rally(0))
            torch.cuda.synchronize()
            t_live = time.perf_counter() - t
            torch.cuda.synchronize()
            t = time.perf_counter()
            want = outcome(lambda: pipe.predict(frames, fps))
            torch.cuda.synchronize()
            t_pred = time.perf_counter() - t
            if got is ValueError or want is ValueError:
                same &= got is want
                refused += got is ValueError
            else:
                same &= bool(torch.equal(got[0], want[0]) and np.array_equal(got[1], want[1]))
            if r:
                live_ms.append(t_live * 1e3)
                predict_ms.append(t_pred * 1e3)
    stat = lambda v: {'median': float(np.median(v)), 'p99': float(np.percentile(v, 99)), 'all': v}
    return {'fps': fps, 'rallies': rallies, 'frames_per_rally': RALLY, 'end_rally_ms': stat(live_ms), 'predict_ms': stat(predict_ms),
            'identical_to_predict': same, 'refused_rallies': refused}


def throughput(pipe, pool, k, rallies):
    with pipe.live(50.0, k=k) as live:
        def run(n):
            for r in range(n):
                for j in range(RALLY):
                    live.push(0, pool[(r * RALLY + j) % len(pool)])
                outcome(lambda: live.end_rally(0))
            torch.cuda.synchronize()
        run(1)
        t = time.perf_counter()
        run(rallies)
        dt = time.perf_counter() - t
    return {'k': k, 'frames': rallies * RALLY, 'frames_per_s': rallies * RALLY / dt}


def paced(pipe, pool, streams, fps, rallies, devices=None, table=None):
    """S cameras at fps, one frame each per tick, rally ends staggered; returns the push lags (s), the push durations (s), the
    end_rally durations (s) and the number of rallies refused with ValueError.  table: every stream's known table, or None."""
    lags, durs, ends, refused = [], [], [], 0
    ticks = rallies * RALLY
    offset = [s * RALLY // streams for s in range(streams)]
    with pipe.live(fps, streams=streams, devices=devices) as live:
        for s in range(streams):
            live.set_table(s, table)
        t0 = time.perf_counter() + 0.05
        for t in range(ticks):
            due = t0 + t / fps
            wait_until(due)
            for s in range(streams):
                a = time.perf_counter()
                live.push(s, pool[(t * streams + s) % len(pool)])
                b = time.perf_counter()
                lags.append(b - due)
                durs.append(b - a)
                if (t + offset[s]) % RALLY == RALLY - 1 or t == ticks - 1:
                    a = time.perf_counter()
                    try:
                        live.end_rally(s)
                    except ValueError:      # a rally predict would refuse: timed like any other
                        refused += 1
                    ends.append(time.perf_counter() - a)
        torch.cuda.synchronize()
    return np.array(lags), np.array(durs), np.array(ends), refused


def max_fps(pipe, pool, streams, devices=None, label=''):
    """The largest fps of LADDER at which `streams` cameras keep to the clock (95th percentile lag below one frame interval)."""
    best, trials = None, []
    for fps in LADDER:
        lags, durs, ends, refused = paced(pipe, pool, streams, fps, 3, devices)
        ok = bool(np.percentile(lags, 95) < 1.0 / fps)
        trials.append({'fps': fps, 'sustained': ok, 'lag_ms_p50': float(np.median(lags) * 1e3),
                       'lag_ms_p95': float(np.percentile(lags, 95) * 1e3), 'lag_ms_max': float(lags.max() * 1e3),
                       'push_ms_p50': float(np.median(durs) * 1e3), 'push_ms_p99': float(np.percentile(durs, 99) * 1e3),
                       'end_rally_ms_median': float(np.median(ends) * 1e3), 'end_rally_ms_p99': float(np.percentile(ends, 99) * 1e3),
                       'refused_rallies': refused})
        print(label, 'streams', streams, json.dumps(trials[-1]), flush=True)
        if not ok:
            break
        best = fps
    return {'per_camera_fps': best, 'ladder': list(LADDER), 'trials': trials}


def cameras_at(pipe, pool, fps, table, most=8):
    """The most cameras (1 .. most) at fps that keep to the clock (95th percentile lag below one frame interval), every stream's
    table set to `table` (None: detected)."""
    best, trials = 0, []
    for streams in range(1, most + 1):
        lags, durs, ends, refused = paced(pipe, pool, streams, fps, 3, table=table)
        ok = bool(np.percentile(lags, 95) < 1.0 / fps)
        trials.append({'cameras': streams, 'sustained': ok, 'lag_ms_p50': float(np.median(lags) * 1e3),
                       'lag_ms_p95': float(np.percentile(lags, 95) * 1e3), 'push_ms_p50': float(np.median(durs) * 1e3),
                       'push_ms_p99': float(np.percentile(durs, 99) * 1e3), 'end_rally_ms_median': float(np.median(ends) * 1e3),
                       'end_rally_ms_p99': float(np.percentile(ends, 99) * 1e3), 'refused_rallies': refused})
        print('known' if table is not None else 'detected', json.dumps(trials[-1]), flush=True)
        if not ok:
            break
        best = streams
    return {'cameras': best, 'fps': fps, 'trials': trials}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True)
    ap.add_argument('--fps', type=float, default=None, help='default 60, or 30 with --known-table')
    ap.add_argument('--rallies', type=int, default=10)
    ap.add_argument('--pipeline', choices=('wasb-hrnet', 'default'), default='wasb-hrnet')
    ap.add_argument('--known-table', action='store_true', help='cameras at --fps with tables set against detected')
    ap.add_argument('--devices', default='', help='comma-separated GPU counts: 1 = the launcher arm, N >= 2 = the scaling arm on N GPUs')
    args = ap.parse_args()
    counts = [int(c) for c in args.devices.split(',') if c]
    if not torch.cuda.is_available():
        raise SystemExit('time_live.py measures on a GPU; none is visible')
    from upliftingtabletennis_b200 import synthetic
    from upliftingtabletennis_b200.interface import TableTennisPipeline
    from upliftingtabletennis_b200.live import DEFAULT_K, DEFAULT_SLOTS
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True, text=True).stdout
    hub = tempfile.mkdtemp(prefix='ttk_live_hub_')
    torch.hub.set_dir(hub)
    write_checkpoints(hub)
    if args.pipeline == 'default':
        write_vitpose_checkpoints(hub)
        pipe = TableTennisPipeline()
        desc = ('default composition: ViTPose main (1152x640, tf32x3) + WASB aux (1280x704, tf32) for the ball, ViTPose main + HRNet aux '
                '(tf32) for the table, uplift (tf32x3); 1080p numpy frames; synthetic weights, on which the two ball detectors disagree')
    else:
        pipe = TableTennisPipeline(ball_model='wasb', ball_model_aux='wasb', table_model='hrnet', table_model_aux='hrnet')
        desc = 'WASB main + aux at 1280x704 (tf32), HRNet main + aux (tf32), uplift (tf32x3); 1080p numpy frames'
    pool = list(synthetic.frames_1080p(128, seed=11))
    result = {'gpus': [l.strip() for l in q.strip().splitlines()], 'default_k': DEFAULT_K, 'default_slots': DEFAULT_SLOTS,
              'pipeline': desc, 'pipeline_arg': args.pipeline}
    if args.known_table:
        frames = pool[:RALLY]
        table = pipe.table_detector.filter_trajectory(pipe.table_detector.predict(frames, return_heatmaps=False)[0],
                                                      pipe.table_detector_aux.predict(frames, return_heatmaps=False)[0])
        fps = args.fps or 30.0
        result['known_table'] = {'visible_keypoints': int(table[:, 2].sum())}
        for label, t in (('detected', None), ('known', table)):           # warm-up of both arms: one camera, one rally
            paced(pipe, pool, 1, fps, 1, table=t)
        for label, t in (('detected', None), ('known', table)):
            result['known_table'][label] = cameras_at(pipe, pool, fps, t)
        result['gpus_after'] = [l.strip() for l in subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                                                                  capture_output=True, text=True).stdout.strip().splitlines()]
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            json.dump(result, f, indent=1)
        return
    args.fps = args.fps or 60.0
    result['latency'] = latency(pipe, pool, args.fps, args.rallies)
    print('latency', json.dumps({k: v for k, v in result['latency'].items()}), flush=True)
    result['k'] = [throughput(pipe, pool, k, 4) for k in (4, 8, 16, 32)]
    print('k', json.dumps(result['k']), flush=True)
    result['max_fps'] = {str(streams): max_fps(pipe, pool, streams) for streams in (1, 2, 4)}
    visible = torch.cuda.device_count()
    skipped = []
    for n in counts:
        if n > visible:
            skipped.append({'gpus': n, 'reason': '%d GPUs visible' % visible})
            continue
        if n == 1:
            result['launcher'] = {
                label: {str(streams): max_fps(pipe, pool, streams, devices, label) for streams in (1, 2, 4)}
                for label, devices in (('devices=None', None), ('devices=[0]', [0]))}
        else:
            arm = result.setdefault('scaling', {})[str(n)] = {}
            for streams in (2, 4, 8, 16):
                if streams < n:                 # a session needs a stream for every entry
                    skipped.append({'gpus': n, 'cameras': streams, 'reason': 'fewer cameras than entries'})
                else:
                    arm[str(streams)] = max_fps(pipe, pool, streams, list(range(n)), 'gpus=%d' % n)
    if counts:
        result['skipped'] = skipped
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(result, f, indent=1)


if __name__ == '__main__':
    main()
